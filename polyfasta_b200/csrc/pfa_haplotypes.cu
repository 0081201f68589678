// Haplotype classes: for every window of this shard (the whole alignment is the single window [0, L)), rep[w][r] = the smallest
// row index whose characters equal row r's over the window's columns of this shard.  Two rows are the same haplotype iff
// K3's d_ij is 0 over those columns: their bits agree at every site K3 marks (the only sites where two rows can differ in the
// planes) and they show the same escape bytes at the same sites.
//
//  0. K3's row-major planes of the marked sites and their sorted site list (pfa_rowmajor_ensure, cached with the alignment);
//     window w of this shard is the local column range [s, e) and the bit range [lo, hi) of the row-major words, found by a
//     binary search over the site list (pfa_hap_windows_kernel).  The exception list is copied once per alignment in row
//     order: (row:24 | site:32 | byte:8) keys, radix-sorted, with an offset per row (pfa_hap_exc_rows_kernel, _offsets_kernel).
//  1. pfa_hap_hash_kernel: a polynomial hash mod 2^64 with an odd base over the row's masked words of [lo, hi) of each plane
//     (16-byte coalesced loads; one warp per chunk of 2,048 words, the chunks of a row add up), plus a mixed term per escape entry
//     (site, byte) in [s, e).
//  2. cub segmented stable sort of (hash -> row), one segment per window: rows stay ascending within equal hashes.
//  3. pfa_hap_verify_kernel: adjacent rows with equal hashes are compared on their contents (words, then escape entries).  A run
//     of equal hashes whose adjacent pairs are all equal is one class whose first row is rep (pfa_hap_rep_kernel, after a max
//     scan gives every position its run's start).  A run with an unequal pair is a hash collision: pfa_hap_split_kernel gives
//     it one warp, which compares every row with the reps found so far in the run.
// The hash is only a sort key: equality is always decided on the contents, so a collision costs time and never a result.
#include <climits>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <cuda/functional>

#include "pfa_common.cuh"

#define PFA_HAP_BASE 0x9E3779B97F4A7C15ull  // odd
#define PFA_HAP_LOW40 ((1ull << 40) - 1ull)  // (site:32 | byte:8) of a row-ordered exception key

// this shard's part of a window: local columns [s, e) and bits [lo, hi) of the row-major words; the hash covers the words
// [a0, a1) of every plane, a0 = (lo / 32) rounded down to a 16-byte boundary, a1 = ceil(hi / 32); bspan = B^(a1 - a0)
struct PfaHapWin {
    int64_t s, e, lo, hi, a0, a1;
    unsigned long long bspan;
};

__device__ __forceinline__ int64_t pfa_hap_lower_bound(const int64_t* __restrict__ a, int64_t n, int64_t x) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ int64_t pfa_hap_lower_bound_u64(const unsigned long long* __restrict__ a, int64_t lo, int64_t hi, unsigned long long x) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ unsigned long long pfa_hap_pow(unsigned long long b, int64_t e) {
    unsigned long long r = 1;
    while (e) {
        if (e & 1) r *= b;
        b *= b;
        e >>= 1;
    }
    return r;
}

// the bits of word j (over marked sites) that lie in [lo, hi)
__device__ __forceinline__ uint32_t pfa_hap_mask(int64_t j, int64_t lo, int64_t hi) {
    const int64_t b = j * 32;
    const int l = (int)(max(lo, b) - b), h = (int)(min(hi, b + 32) - b);
    const uint32_t upper = h >= 32 ? 0xffffffffu : ((1u << h) - 1u);
    return upper & ~((1u << l) - 1u);
}

// the bits of the four words j .. j + 3 that lie in [lo, hi), applied to x (j a multiple of 4)
__device__ __forceinline__ uint4 pfa_hap_mask4(uint4 x, int64_t j, int64_t lo, int64_t hi) {
    const int64_t b = j * 32;
    if (b >= lo && b + 128 <= hi) return x;  // inside the window: every word whole
    const int l = (int)min(max(lo - b, (int64_t)0), (int64_t)128), h = (int)min(max(hi - b, (int64_t)0), (int64_t)128);
    uint32_t v[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {  // bits [l, h) of the 128, as seen from word t
        const int lt = min(max(l - 32 * t, 0), 32), ht = min(max(h - 32 * t, 0), 32);
        const uint32_t upper = ht >= 32 ? 0xffffffffu : ((1u << ht) - 1u), lower = lt >= 32 ? 0xffffffffu : ((1u << lt) - 1u);
        v[t] &= upper & ~lower;
    }
    return make_uint4(v[0], v[1], v[2], v[3]);
}

// row r's entries of the row-ordered exception list at the local columns [s, e)
__device__ __forceinline__ void pfa_hap_exc_range(const unsigned long long* __restrict__ exc, const int64_t* __restrict__ off, int64_t r,
                                                  const PfaHapWin& g, int64_t* e0, int64_t* e1) {
    const int64_t i0 = off[r], i1 = off[r + 1];
    if (i0 == i1 || g.e <= g.s) {
        *e0 = *e1 = i0;
        return;
    }
    const unsigned long long base = (unsigned long long)r << 40;
    *e0 = pfa_hap_lower_bound_u64(exc, i0, i1, base | ((unsigned long long)g.s << 8));
    *e1 = pfa_hap_lower_bound_u64(exc, *e0, i1, base | ((unsigned long long)g.e << 8));
}

__global__ void pfa_hap_windows_kernel(const int64_t* __restrict__ sites, int64_t nsel, int64_t L, int64_t W, int64_t step, int64_t c0,
                                       int64_t ns, int64_t nwin, PfaHapWin* __restrict__ win) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nwin) return;
    const int64_t ws = i * step, we = min(ws + W, L);
    PfaHapWin g;
    g.s = min(max(ws - c0, (int64_t)0), ns);
    g.e = min(max(we - c0, (int64_t)0), ns);
    g.lo = pfa_hap_lower_bound(sites, nsel, g.s);
    g.hi = pfa_hap_lower_bound(sites, nsel, g.e);
    g.a0 = (g.lo >> 5) & ~(int64_t)3;
    g.a1 = g.hi > g.lo ? (g.hi + 31) >> 5 : g.a0;
    g.bspan = pfa_hap_pow(PFA_HAP_BASE, g.a1 - g.a0);
    win[i] = g;
}

// (site:32 | byte:8 | row:24) -> (row:24 | site:32 | byte:8)
__global__ void pfa_hap_exc_rows_kernel(const unsigned long long* __restrict__ keys, int64_t n_exc, unsigned long long* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_exc) return;
    const unsigned long long k = keys[i];
    out[i] = ((k & 0xffffffull) << 40) | ((k >> 32) << 8) | ((k >> 24) & 0xffull);
}

__global__ void pfa_hap_exc_offsets_kernel(const unsigned long long* __restrict__ exc, int64_t n_exc, int64_t n, int64_t* __restrict__ off) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    off[r] = pfa_hap_lower_bound_u64(exc, 0, n_exc, (unsigned long long)r << 40);
}

__global__ void pfa_hap_offsets_kernel(int64_t n, int64_t nwin, int* __restrict__ off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= nwin) off[i] = (int)(i * n);
}

// one warp per (window, row, chunk of PFA_HAP_CHUNK words of every plane): the hash is a sum over word positions, so the chunks of a
// long row add their parts (atomically into zeroed keys when a row has several chunks) and a whole-alignment call keeps every SM
// busy with a few thousand rows.  Lane l reads words 4l .. 4l + 3 of every 128 with one 16-byte load, two loads in flight.
// keys[w n + r] = the row's hash over the window: sum over planes p and words j of word * B^(p (a1 - a0) + j - a0); vals[w n + r] = r
#define PFA_HAP_CHUNK 2048
__global__ void __launch_bounds__(256) pfa_hap_hash_kernel(const uint32_t* __restrict__ rm, int np, int64_t npad, int64_t Wl,
                                                           const PfaHapWin* __restrict__ win, int64_t nwin, int64_t n, int64_t cmax,
                                                           const unsigned long long* __restrict__ exc, const int64_t* __restrict__ exc_off,
                                                           unsigned long long* __restrict__ keys, int* __restrict__ vals) {
    __shared__ unsigned long long blane[32];  // B^(4 lane)
    if (threadIdx.x < 32) blane[threadIdx.x] = pfa_hap_pow(PFA_HAP_BASE, 4 * threadIdx.x);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const unsigned long long b1 = PFA_HAP_BASE, b2 = b1 * b1, b3 = b2 * b1, b128 = pfa_hap_pow(PFA_HAP_BASE, 128), b256 = b128 * b128;
    for (int64_t item = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; item < nwin * n * cmax; item += nwarps) {
        const int64_t wr = cmax == 1 ? item : item / cmax;  // (window, row) < 2^31
        const int c = (int)(item - wr * cmax);
        const int w = (int)((uint32_t)wr / (uint32_t)n), r = (int)((uint32_t)wr - (uint32_t)w * (uint32_t)n);
        const PfaHapWin g = win[w];
        const int64_t c0 = g.a0 + (int64_t)c * PFA_HAP_CHUNK, c1 = min(g.a1, c0 + PFA_HAP_CHUNK);
        if (c > 0 && c0 >= g.a1) continue;  // warp-uniform
        unsigned long long h = 0, bp = c ? pfa_hap_pow(PFA_HAP_BASE, c0 - g.a0) : 1ull;  // B^(p (a1 - a0) + c0 - a0)
        for (int p = 0; p < np; ++p, bp *= g.bspan) {
            const uint32_t* row = rm + ((int64_t)p * npad + r) * Wl;  // 16-byte aligned: Wl is a multiple of 4
            unsigned long long pw = bp * blane[lane];
            int64_t j = c0 + 4 * lane;
            for (; j + 128 < c1; j += 256) {
                const uint4 x = pfa_hap_mask4(__ldg(reinterpret_cast<const uint4*>(row + j)), j, g.lo, g.hi);
                const uint4 y = pfa_hap_mask4(__ldg(reinterpret_cast<const uint4*>(row + j + 128)), j + 128, g.lo, g.hi);
                h += ((unsigned long long)x.x + (unsigned long long)x.y * b1 + (unsigned long long)x.z * b2 + (unsigned long long)x.w * b3) * pw;
                h += ((unsigned long long)y.x + (unsigned long long)y.y * b1 + (unsigned long long)y.z * b2 + (unsigned long long)y.w * b3) * (pw * b128);
                pw *= b256;
            }
            if (j < c1) {  // words beyond a1 are inside the row (a1 <= Wl) and masked off
                const uint4 x = pfa_hap_mask4(__ldg(reinterpret_cast<const uint4*>(row + j)), j, g.lo, g.hi);
                h += ((unsigned long long)x.x + (unsigned long long)x.y * b1 + (unsigned long long)x.z * b2 + (unsigned long long)x.w * b3) * pw;
            }
        }
        if (c == 0) {
            int64_t e0, e1;
            pfa_hap_exc_range(exc, exc_off, r, g, &e0, &e1);
            for (int64_t i = e0 + lane; i < e1; i += 32) {  // splitmix64's finaliser of (site, byte)
                unsigned long long z = (exc[i] & PFA_HAP_LOW40) + 0x9E3779B97F4A7C15ull;
                z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
                z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
                h += z ^ (z >> 31);
            }
        }
        for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
        if (lane == 0) {
            if (cmax == 1) keys[wr] = h;
            else atomicAdd(keys + wr, h);  // exact modulo 2^64
            if (c == 0) vals[wr] = r;
        }
    }
}

// are rows a and b equal over window g?  The whole warp calls it with the same arguments and gets the same answer.
__device__ bool pfa_hap_equal(const uint32_t* __restrict__ rm, int np, int64_t npad, int64_t Wl, const PfaHapWin& g,
                              const unsigned long long* __restrict__ exc, const int64_t* __restrict__ exc_off, int64_t a, int64_t b, int lane) {
    if (a == b) return true;
    if (g.hi > g.lo) {
        const int64_t j0 = g.lo >> 5, j1 = (g.hi + 31) >> 5;
        for (int p = 0; p < np; ++p) {
            const uint32_t* ra = rm + ((int64_t)p * npad + a) * Wl;
            const uint32_t* rb = rm + ((int64_t)p * npad + b) * Wl;
            for (int64_t base = j0; base < j1; base += 32) {  // warp-uniform trip count
                const int64_t j = base + lane;
                const uint32_t d = j < j1 ? (__ldg(ra + j) ^ __ldg(rb + j)) & pfa_hap_mask(j, g.lo, g.hi) : 0u;
                if (__any_sync(0xffffffffu, d != 0)) return false;
            }
        }
    }
    int64_t a0, a1, b0, b1;
    pfa_hap_exc_range(exc, exc_off, a, g, &a0, &a1);
    pfa_hap_exc_range(exc, exc_off, b, g, &b0, &b1);
    if (a1 - a0 != b1 - b0) return false;
    for (int64_t base = 0; base < a1 - a0; base += 32) {
        const int64_t t = base + lane;
        const bool d = t < a1 - a0 && ((exc[a0 + t] ^ exc[b0 + t]) & PFA_HAP_LOW40) != 0;
        if (__any_sync(0xffffffffu, d)) return false;
    }
    return true;
}

// one lane per sorted position i: start[i] = i where a run of equal hashes begins (0 elsewhere, for the max scan); neq[i] = 1 where
// the row differs from the previous one of the same run.  The warp compares the rows of its non-head positions one after the other.
__global__ void __launch_bounds__(256) pfa_hap_verify_kernel(const uint32_t* __restrict__ rm, int np, int64_t npad, int64_t Wl,
                                                             const PfaHapWin* __restrict__ win, int64_t nwin, int64_t n,
                                                             const unsigned long long* __restrict__ exc, const int64_t* __restrict__ exc_off,
                                                             const unsigned long long* __restrict__ keys, const int* __restrict__ vals,
                                                             int* __restrict__ start, uint8_t* __restrict__ neq) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5, N = nwin * n;
    for (int64_t base = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32; base < N; base += nwarps * 32) {
        const int64_t i = base + lane;
        const bool live = i < N;
        const bool head = live && (i % n == 0 || keys[i] != keys[i - 1]);
        unsigned pending = __ballot_sync(0xffffffffu, live && !head);
        bool ne = false;
        while (pending) {  // warp-uniform
            const int src = __ffs(pending) - 1;
            pending &= pending - 1;
            const int64_t ii = base + src;
            const bool eq = pfa_hap_equal(rm, np, npad, Wl, win[ii / n], exc, exc_off, vals[ii - 1], vals[ii], lane);
            if (lane == src) ne = !eq;
        }
        if (live) {
            start[i] = head ? (int)i : 0;
            neq[i] = ne ? 1 : 0;
        }
    }
}

__global__ void pfa_hap_mark_kernel(const int* __restrict__ run, const uint8_t* __restrict__ neq, int64_t N, uint8_t* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N && neq[i]) bad[run[i]] = 1;
}

// runs without an unequal pair: every row's rep is the run's first row; the starts of the other runs are listed for the split
__global__ void pfa_hap_rep_kernel(const int* __restrict__ run, const uint8_t* __restrict__ bad, const int* __restrict__ vals, int64_t N,
                                   int64_t n, int32_t* __restrict__ rep, int* __restrict__ list, int* __restrict__ nlist) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int rs = run[i];
    if (!bad[rs]) rep[(i / n) * n + vals[i]] = vals[rs];
    else if (rs == i) list[atomicAdd(nlist, 1)] = (int)i;
}

// one warp per run with a hash collision: the rows in ascending order, each compared with the reps found so far (marked in
// isrep, which the warp owns for its run's positions)
__global__ void __launch_bounds__(256) pfa_hap_split_kernel(const uint32_t* __restrict__ rm, int np, int64_t npad, int64_t Wl,
                                                            const PfaHapWin* __restrict__ win, int64_t n,
                                                            const unsigned long long* __restrict__ exc, const int64_t* __restrict__ exc_off,
                                                            const int* __restrict__ run, const int* __restrict__ vals,
                                                            const int* __restrict__ list, const int* __restrict__ nlist,
                                                            uint8_t* __restrict__ isrep, int32_t* __restrict__ rep) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t count = *nlist;
    for (int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < count; t += nwarps) {
        const int64_t a = list[t], w = a / n, seg_end = (w + 1) * n;
        const PfaHapWin g = win[w];
        int32_t* rw = rep + w * n;
        for (int64_t i = a; i < seg_end && run[i] == a; ++i) {
            const int r = vals[i];
            int found = -1;
            for (int64_t j = a; j < i && found < 0; ++j)
                if (isrep[j] && pfa_hap_equal(rm, np, npad, Wl, g, exc, exc_off, vals[j], r, lane)) found = vals[j];
            if (lane == 0) {
                isrep[i] = found < 0 ? 1 : 0;
                rw[r] = found < 0 ? r : found;
            }
            __syncwarp();
        }
    }
}

static unsigned pfa_hap_grid(pfa_ctx* ctx, int64_t threads) {
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((threads + 255) / 256, (int64_t)ctx->sm_count * 32));
}

// the row-ordered exception list and its row offsets, built once per alignment
static cudaError_t pfa_exc_rows_ensure(pfa_aln* a) {
    pfa_ctx* ctx = a->ctx;
    if (a->exc_row_off) return cudaSuccess;
    int64_t* off = nullptr;
    cudaError_t e = pfa_dmalloc(ctx, &off, sizeof(int64_t) * (size_t)(a->n + 1));
    if (e != cudaSuccess) return e;
    if (a->n_exc == 0) {
        e = cudaMemsetAsync(off, 0, sizeof(int64_t) * (size_t)(a->n + 1), ctx->stream);
    } else {
        unsigned long long *packed = nullptr, *sorted = nullptr;
        void* tmp = nullptr;
        size_t tmp_bytes = 0;
        const int count = (int)a->n_exc;
        e = pfa_dmalloc(ctx, &packed, sizeof(unsigned long long) * (size_t)count);
        if (e == cudaSuccess) e = pfa_dmalloc(ctx, &sorted, sizeof(unsigned long long) * (size_t)count);
        if (e == cudaSuccess) {
            pfa_hap_exc_rows_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(a->exc_keys, count, packed);
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, packed, sorted, count, 0, 64, ctx->stream);
        if (e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
        if (e == cudaSuccess) e = cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, packed, sorted, count, 0, 64, ctx->stream);
        ctx->launches += 4;
        if (e == cudaSuccess) {
            pfa_hap_exc_offsets_kernel<<<(unsigned)((a->n + 1 + 255) / 256), 256, 0, ctx->stream>>>(sorted, count, a->n, off);
            ctx->launches++;
            e = cudaGetLastError();
        }
        pfa_dfree(ctx, tmp);
        pfa_dfree(ctx, packed);
        if (e == cudaSuccess) a->exc_rows = sorted;
        else pfa_dfree(ctx, sorted);
    }
    if (e == cudaSuccess) a->exc_row_off = off;
    else pfa_dfree(ctx, off);
    return e;
}

extern "C" int pfa_haplotypes_device(pfa_aln* a, int64_t window, int64_t step, int32_t* d_rep) {
    if (!a) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    if (window < 1 || step < 1) return pfa_fail(ctx, PFA_ERR_ARG, "haplotypes: window and step must be >= 1 (got %lld, %lld)", (long long)window, (long long)step);
    const int64_t nwin = pfa_window_count(a->L_total, window, step), n = a->n, N = nwin * n;
    if (N == 0) return PFA_OK;
    if (!d_rep) return pfa_fail(ctx, PFA_ERR_ARG, "haplotypes: null output");
    if (a->ns > INT_MAX) return pfa_fail(ctx, PFA_ERR_ARG, "haplotypes: a shard of more than 2^31-1 sites is not supported");
    if (N > INT_MAX) return pfa_fail(ctx, PFA_ERR_ARG, "haplotypes: %lld windows x %lld rows is more than 2^31-1 classes per call", (long long)nwin, (long long)n);
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    if (a->ns == 0) {  // no column of this shard: one class
        PFA_CUDA(ctx, cudaMemsetAsync(d_rep, 0, sizeof(int32_t) * (size_t)N, ctx->stream));
        return PFA_OK;
    }
    cudaError_t e = pfa_rowmajor_ensure(a);
    if (e == cudaSuccess) e = pfa_exc_rows_ensure(a);
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "haplotypes: row-major planes: %s", cudaGetErrorString(e));
    const int np = a->rowmajor_planes;
    const int64_t npad = (int64_t)a->Wq * 128;
    PfaHapWin* win = nullptr;
    unsigned long long *keys = nullptr, *skeys = nullptr;
    int *vals = nullptr, *svals = nullptr, *off = nullptr, *nlist = nullptr;
    uint8_t *neq = nullptr, *bad = nullptr;
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    e = pfa_dmalloc(ctx, &win, sizeof(PfaHapWin) * (size_t)nwin);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &keys, sizeof(unsigned long long) * (size_t)N);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &skeys, sizeof(unsigned long long) * (size_t)N);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &vals, sizeof(int) * (size_t)N);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &svals, sizeof(int) * (size_t)N);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &off, sizeof(int) * (size_t)(nwin + 1));
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &nlist, sizeof(int));
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &neq, (size_t)N);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &bad, (size_t)N);
    if (e == cudaSuccess) e = cudaMemsetAsync(bad, 0, (size_t)N, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(nlist, 0, sizeof(int), ctx->stream);
    // chunks per (window, row): a window holds at most min(window, ns) marked sites, which span at most that / 32 + 5 words from a0
    const int64_t cmax = (std::min(window, a->ns) / 32 + 5 + PFA_HAP_CHUNK - 1) / PFA_HAP_CHUNK;
    if (e == cudaSuccess && cmax > 1) e = cudaMemsetAsync(keys, 0, sizeof(unsigned long long) * (size_t)N, ctx->stream);
    if (e == cudaSuccess) {
        pfa_hap_windows_kernel<<<(unsigned)((nwin + 255) / 256), 256, 0, ctx->stream>>>(a->rowmajor_sites, a->rowmajor_nsel, a->L_total, window, step,
                                                                                      a->col_begin, a->ns, nwin, win);
        pfa_hap_offsets_kernel<<<(unsigned)((nwin + 1 + 255) / 256), 256, 0, ctx->stream>>>(n, nwin, off);
        pfa_hap_hash_kernel<<<pfa_hap_grid(ctx, N * cmax * 32), 256, 0, ctx->stream>>>(a->rowmajor, np, npad, a->Wl, win, nwin, n, cmax,
                                                                                       a->exc_rows, a->exc_row_off, keys, vals);
        ctx->launches += 3;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess)
        e = cub::DeviceSegmentedSort::StableSortPairs(nullptr, tmp_bytes, keys, skeys, vals, svals, (int)N, (int)nwin, off, off + 1, ctx->stream);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
    if (e == cudaSuccess)
        e = cub::DeviceSegmentedSort::StableSortPairs(tmp, tmp_bytes, keys, skeys, vals, svals, (int)N, (int)nwin, off, off + 1, ctx->stream);
    ctx->launches += 3;
    // after the sort the unsorted buffers are scratch: vals takes the run starts before the scan, keys the scanned starts and the
    // list of runs with a collision
    int* start = vals;
    int* run = reinterpret_cast<int*>(keys);
    int* list = run + N;
    if (e == cudaSuccess) {
        pfa_hap_verify_kernel<<<pfa_hap_grid(ctx, N), 256, 0, ctx->stream>>>(a->rowmajor, np, npad, a->Wl, win, nwin, n, a->exc_rows,
                                                                                  a->exc_row_off, skeys, svals, start, neq);
        ctx->launches++;
        e = cudaGetLastError();
    }
    pfa_dfree(ctx, tmp);
    tmp = nullptr;
    tmp_bytes = 0;
    if (e == cudaSuccess) e = cub::DeviceScan::InclusiveScan(nullptr, tmp_bytes, start, run, ::cuda::maximum<>{}, (int)N, ctx->stream);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
    if (e == cudaSuccess) e = cub::DeviceScan::InclusiveScan(tmp, tmp_bytes, start, run, ::cuda::maximum<>{}, (int)N, ctx->stream);
    ctx->launches++;
    if (e == cudaSuccess) {
        const unsigned g = (unsigned)((N + 255) / 256);
        pfa_hap_mark_kernel<<<g, 256, 0, ctx->stream>>>(run, neq, N, bad);
        pfa_hap_rep_kernel<<<g, 256, 0, ctx->stream>>>(run, bad, svals, N, n, d_rep, list, nlist);
        pfa_hap_split_kernel<<<(unsigned)ctx->sm_count * 8, 256, 0, ctx->stream>>>(a->rowmajor, np, npad, a->Wl, win, n, a->exc_rows, a->exc_row_off,
                                                                                   run, svals, list, nlist, neq, d_rep);
        ctx->launches += 3;
        e = cudaGetLastError();
    }
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, bad);
    pfa_dfree(ctx, neq);
    pfa_dfree(ctx, nlist);
    pfa_dfree(ctx, off);
    pfa_dfree(ctx, svals);
    pfa_dfree(ctx, vals);
    pfa_dfree(ctx, skeys);
    pfa_dfree(ctx, keys);
    pfa_dfree(ctx, win);
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "haplotypes: %s", cudaGetErrorString(e));
    return PFA_OK;
}
