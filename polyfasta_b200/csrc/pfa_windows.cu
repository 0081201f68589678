// Sliding windows along the alignment: S and H of every (population, window) from the per-site H that the site scan stores when
// asked (PfaSiteArgs::hsite), the (columns, D_xy) of every (pair, window) from the divergence scan's per-site values, and the
// PFA_CDS_WIN_LEN-word codon vectors of every (population, window).  The finalisation (pi, theta, D, dxy, ...) is the caller's.
//
// Window i covers the global columns [i step, min(i step + W, L)); windows start at 0, step, 2 step, ... and the first one that
// reaches the end of the alignment is the last (the scikit-allel convention; step > W skips the columns between windows).  Every
// word of a window is a plain integer sum over its columns, so every per-site value is read ONCE whatever W and step are:
//   1. bins of g = gcd(W, step) columns (every window boundary below L is a multiple of g): `words` int64 per (row, bin), laid
//      out [rows][words][nb].  pfa_window_bins_kernel fills two words (non-zero entries, sum) per row of per-site values:
//      bins are cut into pieces of at most PFA_WIN_PIECE columns and a group of lanes per piece sums with coalesced reads, so
//      that the number of lane groups follows rows * ns whatever W and step are (a bin of a whole 10 Mb alignment is 4,883
//      pieces, not one warp); the pieces of a bin that has several add into it atomically (one atomic per piece).  The codon
//      windows' pfa_cds_window_bins_kernel (pfa_codon.cu, next to the codon tables) fills PFA_CDS_WIN_LEN words per bin;
//   2. one in-place exclusive sum over all the bin words (cub);
//   3. each window word is the difference of two prefix sums: O(rows ns + rows words nwin) work whatever W and step are.
// Only the columns of this shard contribute (bins are clipped to the shard), so the vectors of the column shards of an
// alignment add up to the whole alignment's.  All arithmetic is exact int64.
#include <algorithm>

#include <cub/device/device_scan.cuh>

#include "pfa_common.cuh"

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

#define PFA_WIN_PIECE 2048  // columns per piece of a bin: 16 KB of per-site values per warp

// G lanes (a power of two <= 32) per piece; piece m of bin j of row q is item (q nb + j) mpb + m.  bins [rows][2][nb] are zeroed:
// the bin's non-zero count goes to bins[2 q nb + j], its sum nb words further
__global__ void __launch_bounds__(256) pfa_window_bins_kernel(const int64_t* __restrict__ persite, int64_t ns, int64_t c0, int64_t g,
                                                              int64_t b0, int64_t nb, int64_t mpb, int k, int G, int64_t* __restrict__ bins) {
    const int lane = threadIdx.x & 31, sub = lane & (G - 1);
    const int per_warp = 32 / G;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t total = (int64_t)k * nb * mpb;
    for (int64_t base = warp * per_warp; base < total; base += nwarps * per_warp) {  // warp-uniform trip count
        const int64_t e = base + lane / G;
        const int64_t bin = e / mpb;
        int64_t sw = 0;  // the bin's count word
        unsigned long long S = 0, H = 0;
        if (e < total) {
            const int64_t q = bin / nb, j = bin - q * nb, m = e - bin * mpb;
            sw = 2 * q * nb + j;
            const int64_t bs = (b0 + j) * g + m * PFA_WIN_PIECE;  // global columns of the piece, clipped to the bin and the shard
            const int64_t lo = max(c0, bs) - c0, hi = min(min(c0 + ns, (b0 + j + 1) * g), bs + PFA_WIN_PIECE) - c0;
            const int64_t* row = persite + q * ns;
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
                bins[sw] = (int64_t)S;
                bins[sw + nb] = (int64_t)H;
            } else if (S) {  // H > 0 only where S > 0
                atomicAdd(reinterpret_cast<unsigned long long*>(bins + sw), S);
                atomicAdd(reinterpret_cast<unsigned long long*>(bins + sw + nb), H);
            }
        }
    }
}

// counts[(q nwin + i) words + w] = word w of this shard's columns of window i of row q; pre = the exclusive prefix sums of the
// bins [rows][words][nb] (one row of nb bins per (row, word))
__global__ void __launch_bounds__(256) pfa_window_counts_kernel(const int64_t* __restrict__ pre, int64_t L, int64_t W, int64_t step, int64_t g,
                                                                int64_t b0, int64_t nb, int rows, int words, int64_t nwin, int64_t* __restrict__ counts) {
    const int64_t total = (int64_t)rows * nwin * words;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t qi = e / words, w = e - qi * words, q = qi / nwin, i = qi - q * nwin;
        const int64_t ws = i * step, we = min(ws + W, L);
        const int64_t lo = min(max(ws / g - b0, (int64_t)0), nb), hi = min(max((we + g - 1) / g - b0, (int64_t)0), nb);
        const int64_t* row = pre + (q * words + w) * nb;
        counts[e] = hi > lo ? row[hi] - row[lo] : 0;
    }
}

static unsigned pfa_win_grid(pfa_ctx* ctx, int64_t threads) {
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((threads + 255) / 256, (int64_t)ctx->sm_count * 8));
}

// d_counts [rows][nwin][words] from the bins that fill(geometry, bins) adds into a zeroed [rows][words][nb] array
template <typename Fill>
static int pfa_launch_windows(pfa_aln* a, int rows, int words, int64_t window, int64_t step, int64_t* d_counts, Fill fill) {
    pfa_ctx* ctx = a->ctx;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    const int64_t nout = (int64_t)rows * nwin * words;
    if (nout == 0) return PFA_OK;
    const PfaWinGeom w = pfa_win_geom(a, window, step);
    const int64_t nbins = (int64_t)rows * words * w.nb;
    if (nbins == 0) {  // an empty shard contributes nothing
        PFA_CUDA(ctx, cudaMemsetAsync(d_counts, 0, sizeof(int64_t) * (size_t)nout, ctx->stream));
        return PFA_OK;
    }
    int64_t* bins = nullptr;  // scanned in place; the word past the last bin becomes the total
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    cudaError_t e = pfa_dmalloc(ctx, &bins, sizeof(int64_t) * (size_t)(nbins + 1));
    if (e == cudaSuccess) e = cudaMemsetAsync(bins, 0, sizeof(int64_t) * (size_t)(nbins + 1), ctx->stream);
    const int rc = e == cudaSuccess ? fill(w, bins) : PFA_OK;
    if (!rc && e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, bins, nbins + 1, ctx->stream);
    if (!rc && e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
    if (!rc && e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, bins, nbins + 1, ctx->stream);
    if (!rc && e == cudaSuccess) {
        ctx->launches++;
        pfa_window_counts_kernel<<<pfa_win_grid(ctx, nout), 256, 0, ctx->stream>>>(bins, a->L_total, window, step, w.g, w.b0, w.nb, rows, words,
                                                                                   nwin, d_counts);
        ctx->launches++;
        e = cudaGetLastError();
    }
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, bins);
    if (rc) return rc;
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "windows: %s", cudaGetErrorString(e));
    return PFA_OK;
}

int pfa_launch_row_windows(pfa_aln* a, int rows, const int64_t* d_persite, int64_t window, int64_t step, int64_t* d_counts) {
    return pfa_launch_windows(a, rows, 2, window, step, d_counts, [&](const PfaWinGeom& w, int64_t* bins) {
        pfa_ctx* ctx = a->ctx;
        const int64_t mpb = (w.g + PFA_WIN_PIECE - 1) / PFA_WIN_PIECE;  // pieces per bin
        int G = 1;
        while (G < 32 && G < w.g) G *= 2;
        pfa_window_bins_kernel<<<pfa_win_grid(ctx, rows * w.nb * mpb * G), 256, 0, ctx->stream>>>(d_persite, a->ns, a->col_begin, w.g, w.b0, w.nb,
                                                                                                 mpb, rows, G, bins);
        PFA_LAUNCH_CHECK(ctx);
        return PFA_OK;
    });
}

int pfa_launch_cds_windows(pfa_aln* a, const int64_t* d_hsite, const uint8_t* d_labels, int64_t window, int64_t step, int64_t* d_counts) {
    return pfa_launch_windows(a, a->k, PFA_CDS_WIN_LEN, window, step, d_counts, [&](const PfaWinGeom& w, int64_t* bins) {
        return pfa_launch_cds_window_bins(a, d_hsite, d_labels, w.g, w.b0, w.nb, bins);
    });
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
    if (pfa_window_count(a->L_total, window, step) == 0) return PFA_OK;
    if (!d_counts) return pfa_fail(ctx, PFA_ERR_ARG, "windows: null output");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t *d_out = nullptr, *d_hsite = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &d_out, sizeof(int64_t) * (size_t)std::max<int64_t>(pfa_site_len(a), 1)));
    cudaError_t e = pfa_dmalloc(ctx, &d_hsite, sizeof(int64_t) * (size_t)std::max<int64_t>((int64_t)a->k * a->ns, 1));
    if (e != cudaSuccess) {
        pfa_dfree(ctx, d_out);
        return pfa_fail(ctx, PFA_ERR_CUDA, "windows: cudaMallocAsync failed: %s", cudaGetErrorString(e));
    }
    int rc = pfa_launch_site_scan(a, d_out, nullptr, nullptr, false, d_hsite);
    if (!rc) rc = pfa_launch_row_windows(a, a->k, d_hsite, window, step, d_counts);
    pfa_dfree(ctx, d_hsite);
    pfa_dfree(ctx, d_out);
    return rc;
}

}  // extern "C"
