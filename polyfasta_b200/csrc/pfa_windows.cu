// Sliding windows along the alignment: S, H (and through K5 pi, theta, D) of every (population, window) from the per-site H
// that the site scan stores when asked (PfaSiteArgs::hsite).
//
// Window i covers the global columns [i step, min(i step + W, L)); windows start at 0, step, 2 step, ... and the first one that
// reaches the end of the alignment is the last (the scikit-allel convention; step > W skips the columns between windows).  S and
// H of a window are plain integer sums over its columns, so every per-site value is read ONCE whatever W and step are:
//   1. bins of g = gcd(W, step) columns (every window boundary below L is a multiple of g), cut into pieces of at most
//      PFA_WIN_PIECE columns: a group of lanes per piece sums H and counts the non-zero entries (S) with coalesced reads, so
//      that the number of lane groups follows k * ns whatever W and step are (a bin of a whole 10 Mb alignment is 4,883
//      pieces, not one warp); the pieces of a bin that has several add into it atomically (one atomic per piece);
//   2. an exclusive scan over the bins of all populations (cub);
//   3. each window is the difference of two prefix sums.
// Only the columns of this shard contribute (bins are clipped to the shard), so the vectors of the column shards of an
// alignment add up to the whole alignment's.  All arithmetic is exact int64.
// The codon windows (pfa_cds_windows_device) reduce the same way: pfa_cds_window_bins_kernel (pfa_codon.cu, next to the codon
// tables) fills PFA_CDS_WIN_LEN words per (population, bin), one exclusive sum runs over all of them and every window word is
// the difference of two prefix sums: O(k ns + k 72 nwin) work whatever W and step are.
#include <algorithm>
#include <climits>

#include <cub/device/device_scan.cuh>

#include "pfa_common.cuh"

struct PfaSH {
    long long s, h;
};
struct PfaSHAdd {
    __host__ __device__ PfaSH operator()(const PfaSH& a, const PfaSH& b) const { return PfaSH{a.s + b.s, a.h + b.h}; }
};

// the shard's bins: global bin b covers [b g, (b + 1) g); local bin j = global bin b0 + j, clipped to [c0, c0 + ns)
struct PfaWinGeom {
    int64_t g, b0, nb;
};
static PfaWinGeom pfa_win_geom(const pfa_aln* a, int64_t window, int64_t step) {
    int64_t x = window, y = step;
    while (y) {
        const int64_t t = x % y;
        x = y;
        y = t;
    }
    PfaWinGeom w;
    w.g = x;
    w.b0 = a->col_begin / x;
    w.nb = a->ns > 0 ? (a->col_begin + a->ns + x - 1) / x - w.b0 : 0;
    return w;
}

#define PFA_WIN_PIECE 2048  // columns per piece of a bin: 16 KB of per-site H per warp

// G lanes (a power of two <= 32) per piece; piece m of bin j of population q is item (q nb + j) mpb + m.  mpb > 1: the bins
// were zeroed and every piece adds into its bin; mpb == 1: a piece is its whole bin and is stored
__global__ void __launch_bounds__(256) pfa_window_bins_kernel(const int64_t* __restrict__ hsite, int64_t ns, int64_t c0, int64_t g,
                                                              int64_t b0, int64_t nb, int64_t mpb, int k, int G, PfaSH* __restrict__ bins) {
    const int lane = threadIdx.x & 31, sub = lane & (G - 1);
    const int per_warp = 32 / G;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t total = (int64_t)k * nb * mpb;
    for (int64_t base = warp * per_warp; base < total; base += nwarps * per_warp) {  // warp-uniform trip count
        const int64_t e = base + lane / G;
        const int64_t bin = e / mpb;
        unsigned long long S = 0, H = 0;
        if (e < total) {
            const int64_t q = bin / nb, j = bin - q * nb, m = e - bin * mpb;
            const int64_t bs = (b0 + j) * g + m * PFA_WIN_PIECE;  // global columns of the piece, clipped to the bin and the shard
            const int64_t lo = max(c0, bs) - c0, hi = min(min(c0 + ns, (b0 + j + 1) * g), bs + PFA_WIN_PIECE) - c0;
            const int64_t* row = hsite + q * ns;
            int64_t i = lo + sub;
            for (; i + 3 * G < hi; i += 4 * G) {  // four independent loads in flight per lane
                const int64_t h0 = row[i], h1 = row[i + G], h2 = row[i + 2 * G], h3 = row[i + 3 * G];
                H += (unsigned long long)h0 + (unsigned long long)h1 + (unsigned long long)h2 + (unsigned long long)h3;
                S += (h0 != 0 ? 1ull : 0ull) + (h1 != 0 ? 1ull : 0ull) + (h2 != 0 ? 1ull : 0ull) + (h3 != 0 ? 1ull : 0ull);
            }
            for (; i < hi; i += G) {
                const int64_t h = row[i];
                H += (unsigned long long)h;
                S += h != 0 ? 1ull : 0ull;
            }
        }
        for (int off = G / 2; off; off >>= 1) {
            S += __shfl_xor_sync(0xffffffffu, S, off);
            H += __shfl_xor_sync(0xffffffffu, H, off);
        }
        if (e < total && sub == 0) {
            if (mpb == 1) {
                bins[bin] = PfaSH{(long long)S, (long long)H};
            } else if (S) {  // H > 0 only where S > 0
                atomicAdd(reinterpret_cast<unsigned long long*>(&bins[bin].s), S);
                atomicAdd(reinterpret_cast<unsigned long long*>(&bins[bin].h), H);
            }
        }
    }
}

// counts[(q nwin + i) 2 + {0, 1}] = (S, H) of this shard's columns of window i; pre = exclusive prefix sums of the bins
__global__ void __launch_bounds__(256) pfa_window_counts_kernel(const PfaSH* __restrict__ pre, int64_t L, int64_t W, int64_t step, int64_t g,
                                                                int64_t b0, int64_t nb, int k, int64_t nwin, int64_t* __restrict__ counts) {
    const int64_t total = (int64_t)k * nwin;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = e / nwin, i = e - q * nwin;
        const int64_t ws = i * step, we = min(ws + W, L);
        const int64_t lo = min(max(ws / g - b0, (int64_t)0), nb), hi = min(max((we + g - 1) / g - b0, (int64_t)0), nb);
        long long S = 0, H = 0;
        if (hi > lo) {
            S = pre[q * nb + hi].s - pre[q * nb + lo].s;
            H = pre[q * nb + hi].h - pre[q * nb + lo].h;
        }
        counts[2 * e] = S;
        counts[2 * e + 1] = H;
    }
}

// the K5 entries of every (population, window): n of the population, the window's (S, H), seqlen = the window's length
__global__ void __launch_bounds__(256) pfa_window_final_in_kernel(const int64_t* __restrict__ counts, const int64_t* __restrict__ pop_n, int64_t L,
                                                                  int64_t W, int64_t step, int jc, int k, int64_t nwin, pfa_final_in* __restrict__ in) {
    const int64_t total = (int64_t)k * nwin;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = e / nwin, i = e - q * nwin;
        const int64_t ws = i * step, we = min(ws + W, L);
        pfa_final_in p;
        p.n = pop_n[q];
        p.S = counts[2 * e];
        p.H = counts[2 * e + 1];
        p.seqlen = (double)(we - ws);
        p.jc = jc;
        p.pad = 0;
        in[e] = p;
    }
}

static unsigned pfa_win_grid(pfa_ctx* ctx, int64_t threads) {
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((threads + 255) / 256, (int64_t)ctx->sm_count * 8));
}

int pfa_launch_site_windows(pfa_aln* a, const int64_t* d_hsite, int64_t window, int64_t step, int64_t* d_counts) {
    return pfa_launch_row_windows(a, a->k, d_hsite, window, step, d_counts);
}

int pfa_launch_row_windows(pfa_aln* a, int rows, const int64_t* d_persite, int64_t window, int64_t step, int64_t* d_counts) {
    pfa_ctx* ctx = a->ctx;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    const int64_t nout = (int64_t)rows * nwin;
    if (nout == 0) return PFA_OK;
    const PfaWinGeom w = pfa_win_geom(a, window, step);
    const int64_t nbins = (int64_t)rows * w.nb;
    if (nbins == 0) {  // an empty shard contributes nothing
        PFA_CUDA(ctx, cudaMemsetAsync(d_counts, 0, sizeof(int64_t) * 2 * (size_t)nout, ctx->stream));
        return PFA_OK;
    }
    if (nbins + 1 > INT_MAX) return pfa_fail(ctx, PFA_ERR_ARG, "windows: %lld bins of %lld columns exceed the scan's range", (long long)nbins, (long long)w.g);
    const int64_t mpb = (w.g + PFA_WIN_PIECE - 1) / PFA_WIN_PIECE;  // pieces per bin
    PfaSH *bins = nullptr, *pre = nullptr;
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    cudaError_t e = pfa_dmalloc(ctx, &bins, sizeof(PfaSH) * (size_t)(nbins + 1));
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &pre, sizeof(PfaSH) * (size_t)(nbins + 1));
    // the entry past the last bin is the scan's total; with several pieces per bin every bin is a sum of atomics
    if (e == cudaSuccess) e = cudaMemsetAsync(mpb > 1 ? bins : bins + nbins, 0, sizeof(PfaSH) * (size_t)(mpb > 1 ? nbins + 1 : 1), ctx->stream);
    int G = 1;
    while (G < 32 && G < w.g) G *= 2;
    if (e == cudaSuccess) {
        pfa_window_bins_kernel<<<pfa_win_grid(ctx, nbins * mpb * G), 256, 0, ctx->stream>>>(d_persite, a->ns, a->col_begin, w.g, w.b0, w.nb, mpb,
                                                                                           rows, G, bins);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveScan(nullptr, tmp_bytes, bins, pre, PfaSHAdd(), PfaSH{0, 0}, (int)(nbins + 1), ctx->stream);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveScan(tmp, tmp_bytes, bins, pre, PfaSHAdd(), PfaSH{0, 0}, (int)(nbins + 1), ctx->stream);
    if (e == cudaSuccess) {
        ctx->launches++;
        pfa_window_counts_kernel<<<pfa_win_grid(ctx, nout), 256, 0, ctx->stream>>>(pre, a->L_total, window, step, w.g, w.b0, w.nb, rows, nwin, d_counts);
        ctx->launches++;
        e = cudaGetLastError();
    }
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, pre);
    pfa_dfree(ctx, bins);
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "windows: %s", cudaGetErrorString(e));
    return PFA_OK;
}

int pfa_launch_window_final_in(pfa_aln* a, const int64_t* d_counts, int64_t window, int64_t step, int jc, pfa_final_in* d_in) {
    pfa_ctx* ctx = a->ctx;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    const int64_t nout = (int64_t)a->k * nwin;
    if (nout == 0) return PFA_OK;
    pfa_window_final_in_kernel<<<pfa_win_grid(ctx, nout), 256, 0, ctx->stream>>>(d_counts, a->d_pop_n, a->L_total, window, step, jc ? 1 : 0, a->k,
                                                                                  nwin, d_in);
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}

// codon windows: counts[(q nwin + i) PFA_CDS_WIN_LEN + w] = word w of this shard's columns of window i; pre = exclusive prefix
// sums of the bins [k][PFA_CDS_WIN_LEN][nb] (one row of nb bins per (population, word))
__global__ void __launch_bounds__(256) pfa_cds_window_counts_kernel(const long long* __restrict__ pre, int64_t L, int64_t W, int64_t step, int64_t g,
                                                                    int64_t b0, int64_t nb, int k, int64_t nwin, int64_t* __restrict__ counts) {
    const int64_t total = (int64_t)k * nwin * PFA_CDS_WIN_LEN;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t qi = e / PFA_CDS_WIN_LEN, w = e - qi * PFA_CDS_WIN_LEN, q = qi / nwin, i = qi - q * nwin;
        const int64_t ws = i * step, we = min(ws + W, L);
        const int64_t lo = min(max(ws / g - b0, (int64_t)0), nb), hi = min(max((we + g - 1) / g - b0, (int64_t)0), nb);
        const long long* row = pre + (q * PFA_CDS_WIN_LEN + w) * nb;
        counts[e] = hi > lo ? row[hi] - row[lo] : 0;
    }
}

int pfa_launch_cds_windows(pfa_aln* a, const int64_t* d_hsite, const uint8_t* d_labels, int64_t window, int64_t step, int64_t* d_counts) {
    pfa_ctx* ctx = a->ctx;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    const int64_t nout = (int64_t)a->k * nwin;
    if (nout == 0) return PFA_OK;
    const PfaWinGeom w = pfa_win_geom(a, window, step);
    const int64_t nbins = (int64_t)a->k * PFA_CDS_WIN_LEN * w.nb;
    if (nbins == 0) {  // an empty shard contributes nothing
        PFA_CUDA(ctx, cudaMemsetAsync(d_counts, 0, sizeof(int64_t) * PFA_CDS_WIN_LEN * (size_t)nout, ctx->stream));
        return PFA_OK;
    }
    if (nbins + 1 > INT_MAX)
        return pfa_fail(ctx, PFA_ERR_ARG, "cds windows: %lld bin words of %lld columns exceed the scan's range", (long long)nbins, (long long)w.g);
    long long* bins = nullptr;  // scanned in place; the word past the last bin becomes the total
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    cudaError_t e = pfa_dmalloc(ctx, &bins, sizeof(long long) * (size_t)(nbins + 1));
    if (e == cudaSuccess) e = cudaMemsetAsync(bins, 0, sizeof(long long) * (size_t)(nbins + 1), ctx->stream);
    int rc = e == cudaSuccess ? pfa_launch_cds_window_bins(a, d_hsite, d_labels, w.g, w.b0, w.nb, reinterpret_cast<int64_t*>(bins)) : PFA_OK;
    if (!rc && e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, bins, (int)(nbins + 1), ctx->stream);
    if (!rc && e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
    if (!rc && e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, bins, (int)(nbins + 1), ctx->stream);
    if (!rc && e == cudaSuccess) {
        ctx->launches++;
        pfa_cds_window_counts_kernel<<<pfa_win_grid(ctx, nout * PFA_CDS_WIN_LEN), 256, 0, ctx->stream>>>(bins, a->L_total, window, step, w.g, w.b0,
                                                                                                          w.nb, a->k, nwin, d_counts);
        ctx->launches++;
        e = cudaGetLastError();
    }
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, bins);
    if (rc) return rc;
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "cds windows: %s", cudaGetErrorString(e));
    return PFA_OK;
}

extern "C" {

int64_t pfa_window_count(int64_t L, int64_t window, int64_t step) {
    if (L < 0 || window < 1 || step < 1) return -1;
    if (L == 0) return 0;
    const int64_t to_end = 1 + (std::max<int64_t>(0, L - window) + step - 1) / step;  // the first window that reaches L is the last
    const int64_t starts = (L + step - 1) / step;                                       // ... and no window starts at or beyond L
    return std::min(to_end, starts);
}

int pfa_site_windows_device(pfa_aln* a, int64_t window, int64_t step, int64_t* d_counts) {
    if (!a) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    if (window < 1 || step < 1) return pfa_fail(ctx, PFA_ERR_ARG, "windows: window and step must be >= 1 (got %lld, %lld)", (long long)window, (long long)step);
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    if (!d_counts && nwin > 0) return pfa_fail(ctx, PFA_ERR_ARG, "windows: null output");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t *d_out = nullptr, *d_hsite = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &d_out, sizeof(int64_t) * (size_t)std::max<int64_t>(pfa_site_len(a), 1)));
    cudaError_t e = pfa_dmalloc(ctx, &d_hsite, sizeof(int64_t) * (size_t)std::max<int64_t>((int64_t)a->k * a->ns, 1));
    if (e != cudaSuccess) {
        pfa_dfree(ctx, d_out);
        return pfa_fail(ctx, PFA_ERR_CUDA, "windows: cudaMallocAsync failed: %s", cudaGetErrorString(e));
    }
    int rc = pfa_launch_site_scan(a, d_out, nullptr, nullptr, false, d_hsite);
    if (!rc) rc = pfa_launch_site_windows(a, d_hsite, window, step, d_counts);
    pfa_dfree(ctx, d_hsite);
    pfa_dfree(ctx, d_out);
    return rc;
}

int pfa_site_windows(pfa_aln* a, int64_t window, int64_t step, int jc, int64_t* counts, pfa_final_out* fin) {
    if (!a) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    if (window < 1 || step < 1) return pfa_fail(ctx, PFA_ERR_ARG, "windows: window and step must be >= 1 (got %lld, %lld)", (long long)window, (long long)step);
    const int64_t nout = (int64_t)a->k * pfa_window_count(a->L_total, window, step);
    if (nout == 0) return PFA_OK;
    if (!counts) return pfa_fail(ctx, PFA_ERR_ARG, "windows: null output");
    if (fin && nout > INT_MAX) return pfa_fail(ctx, PFA_ERR_ARG, "windows: %lld (population, window) pairs exceed K5's range", (long long)nout);
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t* d_counts = nullptr;
    pfa_final_in* d_in = nullptr;
    pfa_final_out* d_fin = nullptr;
    cudaError_t e = pfa_dmalloc(ctx, &d_counts, sizeof(int64_t) * 2 * (size_t)nout);
    if (e == cudaSuccess && fin) e = pfa_dmalloc(ctx, &d_in, sizeof(pfa_final_in) * (size_t)nout);
    if (e == cudaSuccess && fin) e = pfa_dmalloc(ctx, &d_fin, sizeof(pfa_final_out) * (size_t)nout);
    int rc = e == cudaSuccess ? PFA_OK : pfa_fail(ctx, PFA_ERR_CUDA, "windows: cudaMallocAsync failed: %s", cudaGetErrorString(e));
    if (!rc) rc = pfa_site_windows_device(a, window, step, d_counts);
    if (!rc && fin) rc = pfa_launch_window_final_in(a, d_counts, window, step, jc, d_in);
    if (!rc && fin) rc = pfa_launch_finalize(ctx, d_in, d_fin, (int)nout);
    if (!rc) {
        e = cudaMemcpyAsync(counts, d_counts, sizeof(int64_t) * 2 * (size_t)nout, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess && fin) e = cudaMemcpyAsync(fin, d_fin, sizeof(pfa_final_out) * (size_t)nout, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "windows: result copy failed: %s", cudaGetErrorString(e));
    }
    pfa_dfree(ctx, d_fin);
    pfa_dfree(ctx, d_in);
    pfa_dfree(ctx, d_counts);
    return rc;
}

}  // extern "C"
