// K1: text -> site-major bit-planes (GPU side of ingest), exception list, synthetic generator.
//
// Replaces the in-memory form readfasta (PolyFastA.py:227-250) hands to the scans: instead of n Python
// strings the alignment lives in HBM as three bit-planes over ROWS, one record per SITE, so that the
// per-column allele counts of getvarsites (PolyFastA.py:252-261) become popcounts of ANDed words.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "pfa_common.cuh"
#include "pfa_synth.cuh"

// symbol -> 4-bit code: bit0 b0, bit1 b1, bit2 v (valid ACGT), bit3 escape (byte kept in the exception list).
// Lower case folds onto upper case (readfasta upper-cases, PolyFastA.py:236,245).
__device__ __forceinline__ unsigned classify_byte(unsigned c) {
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

// One warp = 32 rows (one 32-bit word of every plane) x 32 consecutive sites.  Lane j reads 32 bytes of
// row 32*w+j (a full sector), the 32 sites are transposed with ballots, lane s writes the words of site s.
__global__ void __launch_bounds__(256) pfa_encode_kernel(const uint8_t* __restrict__ text, int64_t ldt, int64_t n,
                                                         int64_t cols, int64_t site0, uint32_t* __restrict__ b0,
                                                         uint32_t* __restrict__ b1, uint32_t* __restrict__ v, int Wn,
                                                         unsigned long long* __restrict__ exc_keys,
                                                         unsigned long long* __restrict__ exc_count, int64_t exc_cap,
                                                         int* __restrict__ has_invalid, int vec_ok, uint32_t* __restrict__ vflag, int gc) {
    __shared__ uint8_t lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = (uint8_t)classify_byte(i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t sg = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // group of 32 sites
    const int64_t w = blockIdx.y;                                                      // word index over rows
    const int64_t c0 = sg * 32;
    if (c0 >= cols) return;
    const int64_t row = w * 32 + lane;
    uint32_t bytes[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) bytes[i] = 0x2d2d2d2du;  // '-' : code 0, same as the padding rows
    const bool live = row < n;
    if (live) {
        const uint8_t* src = text + row * ldt + c0;
        if (vec_ok && c0 + 32 <= cols) {
            const uint4* s4 = reinterpret_cast<const uint4*>(src);
            uint4 a = __ldg(s4), b = __ldg(s4 + 1);
            bytes[0] = a.x; bytes[1] = a.y; bytes[2] = a.z; bytes[3] = a.w;
            bytes[4] = b.x; bytes[5] = b.y; bytes[6] = b.z; bytes[7] = b.w;
        } else {
            const int lim = (int)min((int64_t)32, cols - c0);
            for (int i = 0; i < lim; ++i) {
                uint32_t c = src[i];
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
        const bool in_range = c0 + s < cols;
        if (live && in_range && !(code & 4u)) any_invalid = true;
        if (live && in_range && (code & 8u)) {
            const unsigned up = (c >= 'a' && c <= 'z') ? c - 32 : c;
            const unsigned long long slot = atomicAdd(exc_count, 1ull);
            if ((int64_t)slot < exc_cap)
                exc_keys[slot] = ((unsigned long long)(site0 + c0 + s) << 32) | ((unsigned long long)up << 24) |
                                 (unsigned long long)row;
        }
    }
    if (__any_sync(0xffffffffu, any_invalid) && lane == 0) atomicOr(has_invalid, 1);
    const uint32_t wlive = __ballot_sync(0xffffffffu, live);
    if (c0 + lane < cols) {
        const int64_t o = (site0 + c0 + lane) * (int64_t)Wn + w;
        b0[o] = my0; b1[o] = my1; v[o] = myv;
        if (myv != wlive) atomicOr(vflag + site0 + c0 + lane, 1u << (int)((w >> 2) / gc));  // this 128-row chunk holds a non-ACGT symbol
    }
}

int pfa_encode_chunk(pfa_aln* a, const uint8_t* d_text, int64_t ldt, int64_t cols, int64_t site0,
                     unsigned long long* d_exc_count, int64_t exc_cap, int* d_has_invalid, cudaStream_t st) {
    pfa_ctx* ctx = a->ctx;
    if (cols <= 0 || a->n <= 0) return PFA_OK;
    if (!st) st = ctx->stream;
    const int64_t groups = (cols + 31) / 32;
    const int vec_ok = (reinterpret_cast<uintptr_t>(d_text) % 16 == 0) && (ldt % 16 == 0);
    dim3 grid((unsigned)((groups + 7) / 8), (unsigned)((a->n + 31) / 32));
    pfa_encode_kernel<<<grid, 256, 0, st>>>(d_text, ldt, a->n, cols, site0, (uint32_t*)a->b0, (uint32_t*)a->b1,
                                                     (uint32_t*)a->v, a->Wq * 4, a->exc_keys, d_exc_count, exc_cap,
                                                     d_has_invalid, vec_ok, a->vflag, a->gc);
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}

// Same transposition for a chunk the HOST has packed (pfa_pack.cpp): 4 bases per byte, optionally one validity bit per base.
// One warp = 32 rows x 64 sites: lane j reads 16 bytes of codes (and 8 bytes of validity) of row 32*w+j.
//   direct = 0: codes t = A 0, C 1, T 2, G 3 of the ACGT-only packer (b1 = t1, b0 = t0 ^ t1), every base valid;
//   direct = 1: codes already as the planes want them (A0 C1 G2 T3 / '-'0 'N'1 '?'2); valid == nullptr: every base valid.
template <bool HAS_VALID, bool DIRECT>
__global__ void __launch_bounds__(256) pfa_encode_packed_kernel(const uint8_t* __restrict__ packed, int64_t ldp,
                                                                const uint8_t* __restrict__ valid, int64_t ldv,
                                                                int64_t n, int64_t cols, int64_t site0, uint32_t* __restrict__ b0,
                                                                uint32_t* __restrict__ b1, uint32_t* __restrict__ v, int Wn,
                                                                int* __restrict__ has_invalid, uint32_t* __restrict__ vflag, int gc) {
    const int lane = threadIdx.x & 31;
    const int64_t sg = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // group of 64 sites
    const int64_t w = blockIdx.y;
    const int64_t c0 = sg * 64;
    if (c0 >= cols) return;
    const int64_t row = w * 32 + lane;
    const bool live = row < n;
    uint4 x = make_uint4(0, 0, 0, 0);
    uint2 vb = live ? make_uint2(0xffffffffu, 0xffffffffu) : make_uint2(0u, 0u);
    if (live) {
        x = __ldg(reinterpret_cast<const uint4*>(packed + row * ldp + (c0 >> 2)));
        if (HAS_VALID) vb = __ldg(reinterpret_cast<const uint2*>(valid + row * ldv + (c0 >> 3)));
    }
    const uint32_t wlive = __ballot_sync(0xffffffffu, live);
    const uint32_t words[4] = {x.x, x.y, x.z, x.w};
    const uint32_t vwords[2] = {vb.x, vb.y};
    bool any_invalid = false;
#pragma unroll
    for (int h = 0; h < 2; ++h) {  // sites c0 + 32h + s
        uint32_t my0 = 0, my1 = 0, myv = 0;
#pragma unroll
        for (int s = 0; s < 32; ++s) {
            const uint32_t t = (words[2 * h + (s >> 4)] >> (2 * (s & 15))) & 3u;
            const uint32_t w1 = __ballot_sync(0xffffffffu, t & 2u);
            const uint32_t w0 = __ballot_sync(0xffffffffu, (DIRECT ? t : (t ^ (t >> 1))) & 1u);
            uint32_t wv = wlive;
            if (HAS_VALID) wv = __ballot_sync(0xffffffffu, (vwords[h] >> s) & 1u);
            if (lane == s) { my0 = w0; my1 = w1; myv = wv; }
        }
        const int64_t c = c0 + 32 * h + lane;
        if (c < cols) {
            const int64_t o = (site0 + c) * (int64_t)Wn + w;
            b0[o] = my0; b1[o] = my1; v[o] = myv;
            if (myv != wlive) {
                any_invalid = true;
                atomicOr(vflag + site0 + c, 1u << (int)((w >> 2) / gc));
            }
        }
    }
    if (HAS_VALID && __any_sync(0xffffffffu, any_invalid) && lane == 0) atomicOr(has_invalid, 1);
}

int pfa_encode_packed_chunk(pfa_aln* a, const uint8_t* d_packed, int64_t ldp, const uint8_t* d_valid, int64_t ldv, int direct,
                            int64_t cols, int64_t site0, int* d_has_invalid, cudaStream_t st) {
    pfa_ctx* ctx = a->ctx;
    if (cols <= 0 || a->n <= 0) return PFA_OK;
    if (ldp % 16 != 0 || reinterpret_cast<uintptr_t>(d_packed) % 16 != 0 || ldp * 4 < pfa_round_up(cols, 64) ||
        (d_valid && (ldv % 8 != 0 || reinterpret_cast<uintptr_t>(d_valid) % 8 != 0 || ldv * 8 < pfa_round_up(cols, 64))))
        return pfa_fail(ctx, PFA_ERR_ARG, "packed chunk: rows must be 16-byte aligned and padded to 64 bases");
    const int64_t groups = (cols + 63) / 64;
    dim3 grid((unsigned)((groups + 7) / 8), (unsigned)((a->n + 31) / 32));
#define PFA_PACKED_LAUNCH(V_, D_)                                                                                     \
    pfa_encode_packed_kernel<V_, D_><<<grid, 256, 0, st>>>(d_packed, ldp, d_valid, ldv, a->n, cols, site0, (uint32_t*)a->b0,    \
                                                           (uint32_t*)a->b1, (uint32_t*)a->v, a->Wq * 4, d_has_invalid, a->vflag, a->gc)
    if (d_valid && direct) PFA_PACKED_LAUNCH(true, true);
    else if (d_valid) PFA_PACKED_LAUNCH(true, false);
    else if (direct) PFA_PACKED_LAUNCH(false, true);
    else PFA_PACKED_LAUNCH(false, false);
#undef PFA_PACKED_LAUNCH
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}

// ---- exception list: sort by (site, byte, row), then the first index of every distinct site -------------
__global__ void pfa_head_flags_kernel(const unsigned long long* __restrict__ keys, int64_t n, uint8_t* __restrict__ flags) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = (i == 0) || ((keys[i] >> 32) != (keys[i - 1] >> 32));
}

// sorts `count` keys in place (the buffer is replaced) and returns the index of the first key of every distinct site
int pfa_sort_exceptions(pfa_ctx* ctx, unsigned long long** keys, int64_t count, int64_t** heads_out, int64_t* n_heads) {
    *heads_out = nullptr;
    *n_heads = 0;
    if (count == 0) return PFA_OK;
    unsigned long long* sorted = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &sorted, sizeof(unsigned long long) * (size_t)count));
    size_t tmp_bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, *keys, sorted, (int)count, 0, 64, ctx->stream);
    void* tmp = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &tmp, tmp_bytes));
    PFA_CUDA(ctx, cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, *keys, sorted, (int)count, 0, 64, ctx->stream));
    ctx->launches += 4;
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, *keys);
    *keys = sorted;

    uint8_t* flags = nullptr;
    int64_t* d_num = nullptr;
    int64_t* heads = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &flags, (size_t)count));
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &heads, sizeof(int64_t) * (size_t)count));
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &d_num, sizeof(int64_t)));
    pfa_head_flags_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(sorted, count, flags);
    PFA_LAUNCH_CHECK(ctx);
    cub::CountingInputIterator<int64_t> idx(0);
    tmp_bytes = 0;
    cub::DeviceSelect::Flagged(nullptr, tmp_bytes, idx, flags, heads, d_num, (int)count, ctx->stream);
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &tmp, tmp_bytes));
    PFA_CUDA(ctx, cub::DeviceSelect::Flagged(tmp, tmp_bytes, idx, flags, heads, d_num, (int)count, ctx->stream));
    ctx->launches += 2;
    int64_t num = 0;
    PFA_CUDA(ctx, cudaMemcpyAsync(&num, d_num, sizeof(num), cudaMemcpyDeviceToHost, ctx->stream));
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, flags);
    pfa_dfree(ctx, d_num);
    *heads_out = heads;
    *n_heads = num;
    return PFA_OK;
}

int pfa_finish_exceptions(pfa_aln* a, int64_t count) {
    a->n_exc = count;
    a->n_exc_sites = 0;
    return pfa_sort_exceptions(a->ctx, &a->exc_keys, count, &a->exc_heads, &a->n_exc_sites);
}

// ---- synthetic generator: the planes of columns [col_begin, col_begin+ns) written directly ---------------
// One thread per (site, 32-row word).  Monomorphic sites are constant words; segregating sites evaluate the
// row permutation (A*r + B) mod n per row.  polyfasta_b200/synth.py is the numpy twin of pfa_synth.cuh.
__global__ void __launch_bounds__(256) pfa_synth_kernel(uint32_t* __restrict__ b0, uint32_t* __restrict__ b1,
                                                        uint32_t* __restrict__ v, int64_t ns, int64_t col_begin, int64_t n,
                                                        int Wn, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm,
                                                        uint64_t mult) {
    const int nwords = (int)((n + 31) / 32);
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t site = t / nwords;
    const int w = (int)(t % nwords);
    if (site >= ns) return;
    const pfa_synth_site sp = pfa_synth_site_params(seed, (uint64_t)(col_begin + site), (uint64_t)n, p_seg_ppm, tri_ppm);
    const int rows_here = (int)min((int64_t)32, n - (int64_t)w * 32);
    const uint32_t live = rows_here == 32 ? 0xffffffffu : ((1u << rows_here) - 1u);
    uint32_t w0, w1;
    if (!sp.k1) {
        w0 = (sp.anc & 1) ? live : 0u;
        w1 = (sp.anc & 2) ? live : 0u;
    } else {
        w0 = w1 = 0;
        for (int i = 0; i < rows_here; ++i) {
            const uint32_t base = pfa_synth_base(sp, (uint64_t)w * 32 + i, (uint64_t)n, mult);
            w0 |= (base & 1u) << i;
            w1 |= ((base >> 1) & 1u) << i;
        }
    }
    const int64_t o = site * (int64_t)Wn + w;
    b0[o] = w0; b1[o] = w1; v[o] = live;
}

int pfa_synth_fill(pfa_aln* a, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm) {
    pfa_ctx* ctx = a->ctx;
    const int64_t nwords = (a->n + 31) / 32;
    const int64_t total = a->ns * nwords;
    if (total == 0) return PFA_OK;
    const uint64_t mult = pfa_synth_multiplier((uint64_t)a->n);
    // launch in slices of whole sites so that gridDim.x stays below 2^31
    const int64_t sites_per_launch = std::max<int64_t>(1, ((int64_t)1 << 30) / nwords);
    for (int64_t site_lo = 0; site_lo < a->ns; site_lo += sites_per_launch) {
        const int64_t site_hi = std::min<int64_t>(a->ns, site_lo + sites_per_launch);
        const int64_t cnt = (site_hi - site_lo) * nwords;
        const int64_t off = site_lo * (int64_t)a->Wq * 4;
        pfa_synth_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, ctx->stream>>>(
            (uint32_t*)a->b0 + off, (uint32_t*)a->b1 + off, (uint32_t*)a->v + off, site_hi - site_lo,
            a->col_begin + site_lo, a->n, a->Wq * 4, seed, p_seg_ppm, tri_ppm, mult);
        PFA_LAUNCH_CHECK(ctx);
    }
    return PFA_OK;
}

// sparse gaps poked into the planes of an alignment (benchmarks and tests of the validity flags): see pfa_synth_gap_bit
__global__ void __launch_bounds__(256) pfa_poke_gaps_kernel(uint32_t* __restrict__ b0, uint32_t* __restrict__ b1, uint32_t* __restrict__ v,
                                                            uint32_t* __restrict__ vflag, int gc, int64_t ns, int64_t col_begin, int64_t n, int Wn,
                                                            uint64_t seed, uint32_t gap_ppm, int* __restrict__ any) {
    const int nwords = (int)((n + 31) / 32);
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t site = t / nwords;
    const int w = (int)(t % nwords);
    if (site >= ns) return;
    const uint32_t bit = pfa_synth_gap_bit(seed, (uint64_t)(col_begin + site), (uint64_t)w, gap_ppm);
    if (bit >= 32u || (int64_t)w * 32 + bit >= n) return;
    const int64_t o = site * (int64_t)Wn + w;
    b0[o] &= ~(1u << bit);
    b1[o] &= ~(1u << bit);
    v[o] &= ~(1u << bit);
    atomicOr(vflag + site, 1u << ((w >> 2) / gc));
    *any = 1;
}

extern "C" int pfa_aln_poke_gaps(pfa_aln* a, uint64_t seed, uint32_t gap_ppm) {
    if (!a || gap_ppm > 31250u) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t nwords = (a->n + 31) / 32;
    if (a->ns == 0 || nwords == 0 || gap_ppm == 0) return PFA_OK;
    int* d_any = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &d_any, sizeof(int)));
    PFA_CUDA(ctx, cudaMemsetAsync(d_any, 0, sizeof(int), ctx->stream));
    const int64_t sites_per_launch = std::max<int64_t>(1, ((int64_t)1 << 30) / nwords);
    for (int64_t site_lo = 0; site_lo < a->ns; site_lo += sites_per_launch) {
        const int64_t site_hi = std::min<int64_t>(a->ns, site_lo + sites_per_launch);
        const int64_t cnt = (site_hi - site_lo) * nwords;
        const int64_t off = site_lo * (int64_t)a->Wq * 4;
        pfa_poke_gaps_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, ctx->stream>>>((uint32_t*)a->b0 + off, (uint32_t*)a->b1 + off, (uint32_t*)a->v + off,
                                                                                   a->vflag + site_lo, a->gc, site_hi - site_lo, a->col_begin + site_lo,
                                                                                   a->n, a->Wq * 4, seed, gap_ppm, d_any);
        PFA_LAUNCH_CHECK(ctx);
    }
    int any = 0;
    PFA_CUDA(ctx, cudaMemcpyAsync(&any, d_any, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    pfa_dfree(ctx, d_any);
    if (any) a->has_invalid |= 1;
    a->vflag_sites = -1;  // recount on the next sparse scan
    if (a->rowmajor) {  // the pairwise kernel's transposed copy is stale
        pfa_dfree(ctx, a->rowmajor);
        pfa_dfree(ctx, a->rowmajor_sites);
        a->rowmajor = nullptr;
        a->rowmajor_sites = nullptr;
        a->rowmajor_nsel = 0;
    }
    return PFA_OK;
}

// the same synthetic alignment as upper-case text in device memory (input of the end-to-end benchmark leg):
// one thread writes 16 consecutive sites of one row
__global__ void __launch_bounds__(256) pfa_synth_text_kernel(uint8_t* __restrict__ text, int64_t ld, int64_t n, int64_t cols,
                                                             int64_t col_begin, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm,
                                                             uint64_t mult) {
    const int64_t groups = (cols + 15) / 16;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t row = t / groups, g = t % groups;
    if (row >= n) return;
    uint8_t out[16];
    const int64_t c0 = g * 16;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const pfa_synth_site sp = pfa_synth_site_params(seed, (uint64_t)(col_begin + c0 + i), (uint64_t)n, p_seg_ppm, tri_ppm);
        const uint32_t b = sp.k1 ? pfa_synth_base(sp, (uint64_t)row, (uint64_t)n, mult) : sp.anc;
        out[i] = (uint8_t)("ACGT"[b]);
    }
    uint8_t* dst = text + row * ld + c0;
    if (c0 + 16 <= cols && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(out);
    } else {
        for (int i = 0; i < 16 && c0 + i < cols; ++i) dst[i] = out[i];
    }
}

extern "C" int pfa_synth_text_device(pfa_ctx* ctx, uint8_t* d_text, int64_t ld, int64_t n, uint64_t seed, uint32_t p_seg_ppm,
                                     uint32_t tri_ppm, int64_t col_begin, int64_t col_end) {
    if (!ctx || !d_text || n <= 0 || col_end < col_begin || ld < col_end - col_begin) return PFA_ERR_ARG;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t cols = col_end - col_begin;
    if (!cols) return PFA_OK;
    const int64_t groups = (cols + 15) / 16;
    const int64_t blocks = (n * groups + 255) / 256;
    if (blocks >= ((int64_t)1 << 31)) return pfa_fail(ctx, PFA_ERR_ARG, "synthetic text: n * cols too large for one launch");
    pfa_synth_text_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(d_text, ld, n, cols, col_begin, seed, p_seg_ppm, tri_ppm,
                                                                     pfa_synth_multiplier((uint64_t)n));
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}
