// Divergence between populations (beyond the reference): d_xy, net divergence d_a and Hudson's F_ST for every pair x < y of
// the populations, over the whole alignment and in sliding windows.
//
// Every character is an allele (PolyFastA.py:256-258).  For populations X, Y and a column c with class counts c_{X,a}:
//   Dxy_site(c) = n_x n_y - sum_a c_{X,a} c_{Y,a}
// = the number of ordered row pairs (i in X, j in Y) whose characters differ at c (a row in both populations compares equal to
// itself).  D_xy = sum_c Dxy_site(c) is an exact int64 that column shards add up; floats appear only in the finalisation.
//   0. pfa_launch_var_flags (K3's first step, pfa_pairwise.cu) marks the sites at which two rows differ in the planes;
//      cub::DeviceSelect lists them.  No other site has a non-zero Dxy_site, except sites where only escape BYTES differ.
//   1. pfa_divergence_kernel<HAS_V>: one warp per listed site.  Class counts per population (pfa_class_counts), per-pair
//      cross terms from the lanes, per-pair totals in registers / shared memory, one global atomic per block and pair.
//      A site where some population has an escape row is left to step 2, so nothing is counted twice.
//   2. pfa_divergence_escape_kernel: one warp per site of the exception list where some population has an escape row.  The
//      keys of a site are sorted by (byte, row): each run of one byte adds e_x e_y to the cross term.  This also covers
//      columns where every row is an escape row but the bytes differ, which step 0 does not mark.
//   3. windows: the per-site values (P rows of ns) go through the window reduction of pfa_windows.cu.
//   4. pfa_div_finalize_kernel: dxy, d_a, F_ST in fp64 with round-to-nearest intrinsics (-fmad=false for the library).
#include <algorithm>
#include <climits>

#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "pfa_common.cuh"
#include "pfa_sites.cuh"

#define PFA_DIV_MAX_POPS 64  // per-warp class counts (8 x 64 x 8 x 4 B) and per-block pair sums (2,016 x 8 B) in shared memory
#define PFA_DIV_MAX_PAIRS (PFA_DIV_MAX_POPS * (PFA_DIV_MAX_POPS - 1) / 2)
#define PFA_DIV_WARPS 8
#define PFA_DIV_GAP 7  // slot of the gap class next to the seven packed classes

// pair p -> (x, y), x < y, in the order (0,1), (0,2), ..., (0,k-1), (1,2), ...
__device__ __forceinline__ void pfa_div_pair_table(int k, uint8_t* px, uint8_t* py) {
    for (int x = threadIdx.x; x < k; x += blockDim.x) {
        const int base = x * (2 * k - x - 1) / 2;
        for (int y = x + 1; y < k; ++y) {
            px[base + y - x - 1] = (uint8_t)x;
            py[base + y - x - 1] = (uint8_t)y;
        }
    }
}

// class counts of every population at site s into cw[q][0..7] (slot 7: gap = n_q - the seven packed classes); returns true
// when some population has an escape row there
template <bool HAS_V>
__device__ __forceinline__ bool pfa_div_counts(const uint4* __restrict__ b0, const uint4* __restrict__ b1, const uint4* __restrict__ v,
                                               const uint4* __restrict__ masks, int Wq, const int64_t* __restrict__ pop_n, int k,
                                               int64_t s, int lane, uint32_t (*cw)[8]) {
    const uint4 *p0 = b0 + s * Wq, *p1 = b1 + s * Wq, *pv = v + s * Wq;
    bool esc = false;
    for (int q = 0; q < k; ++q) {
        uint32_t c[PFA_NCLASS];
        pfa_class_counts<HAS_V>(p0, p1, pv, masks + (int64_t)q * Wq, Wq, lane, c);
        uint32_t sum = 0;
#pragma unroll
        for (int i = 0; i < PFA_NCLASS; ++i) sum += HAS_V || i < 4 ? c[i] : 0u;
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < PFA_NCLASS; ++i) cw[q][i] = HAS_V || i < 4 ? c[i] : 0u;
            cw[q][PFA_DIV_GAP] = (uint32_t)pop_n[q] - sum;
        }
        esc |= HAS_V && c[PFA_C_ESC] != 0;  // warp-uniform
    }
    __syncwarp();
    return esc;
}

// n_x n_y - sum over A, C, G, T, N, ?, gap of c_x c_y (the escape class is left out: its bytes decide)
__device__ __forceinline__ unsigned long long pfa_div_plane_d(const uint32_t* cx, const uint32_t* cy, const int64_t* __restrict__ pop_n, int x, int y) {
    unsigned long long cross = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (i != PFA_C_ESC) cross += (unsigned long long)cx[i] * cy[i];
    return (unsigned long long)pop_n[x] * (unsigned long long)pop_n[y] - cross;
}

// one warp per listed site; out[p] += D of pair p, dsite[p ns + s] = Dxy_site (optional, zero-filled by the launch)
template <bool HAS_V>
__global__ void __launch_bounds__(256) pfa_divergence_kernel(const uint4* __restrict__ b0, const uint4* __restrict__ b1, const uint4* __restrict__ v,
                                                             const uint4* __restrict__ masks, int Wq, const int64_t* __restrict__ pop_n, int k,
                                                             const int64_t* __restrict__ sites, const int64_t* __restrict__ nsel, int64_t ns,
                                                             unsigned long long* __restrict__ out, int64_t* __restrict__ dsite) {
    __shared__ uint32_t cnt[PFA_DIV_WARPS][PFA_DIV_MAX_POPS][8];
    __shared__ unsigned long long tot[PFA_DIV_MAX_PAIRS];
    __shared__ uint8_t px[PFA_DIV_MAX_PAIRS], py[PFA_DIV_MAX_PAIRS];
    const int P = k * (k - 1) / 2;
    for (int p = threadIdx.x; p < P; p += blockDim.x) tot[p] = 0ull;
    pfa_div_pair_table(k, px, py);
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t nwarps = (int64_t)gridDim.x * PFA_DIV_WARPS;
    const int64_t m = *nsel;
    unsigned long long acc = 0;  // pair `lane` (the pairs from 32 on add into shared memory site by site)
    for (int64_t i = (int64_t)blockIdx.x * PFA_DIV_WARPS + wib; i < m; i += nwarps) {
        const int64_t s = sites[i];
        if (pfa_div_counts<HAS_V>(b0, b1, v, masks, Wq, pop_n, k, s, lane, cnt[wib])) continue;  // pfa_divergence_escape_kernel
        for (int p = lane; p < P; p += 32) {
            const unsigned long long d = pfa_div_plane_d(cnt[wib][px[p]], cnt[wib][py[p]], pop_n, px[p], py[p]);
            if (p < 32) acc += d;
            else if (d) atomicAdd(&tot[p], d);
            if (dsite && d) dsite[(int64_t)p * ns + s] = (int64_t)d;
        }
        __syncwarp();
    }
    if (lane < P && acc) atomicAdd(&tot[lane], acc);
    __syncthreads();
    for (int p = threadIdx.x; p < P; p += blockDim.x)
        if (tot[p]) atomicAdd(out + p, tot[p]);
}

// one warp per site of the exception list at which some population has an escape row: the plane classes as above, and for
// every run of one escape byte (keys sorted by site, byte, row) e_x e_y more pairs that compare equal
__global__ void __launch_bounds__(256) pfa_divergence_escape_kernel(const uint4* __restrict__ b0, const uint4* __restrict__ b1,
                                                                    const uint4* __restrict__ v, const uint4* __restrict__ masks, int Wq,
                                                                    const int64_t* __restrict__ pop_n, int k,
                                                                    const unsigned long long* __restrict__ keys, int64_t n_exc,
                                                                    const int64_t* __restrict__ heads, int64_t n_heads, int64_t ns,
                                                                    unsigned long long* __restrict__ out, int64_t* __restrict__ dsite) {
    __shared__ uint32_t cnt[PFA_DIV_WARPS][PFA_DIV_MAX_POPS][8];
    __shared__ uint32_t run[PFA_DIV_WARPS][PFA_DIV_MAX_POPS];
    __shared__ unsigned long long tot[PFA_DIV_MAX_PAIRS];
    __shared__ uint8_t px[PFA_DIV_MAX_PAIRS], py[PFA_DIV_MAX_PAIRS];
    const int P = k * (k - 1) / 2;
    for (int p = threadIdx.x; p < P; p += blockDim.x) tot[p] = 0ull;
    pfa_div_pair_table(k, px, py);
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t nwarps = (int64_t)gridDim.x * PFA_DIV_WARPS;
    const int Wn = Wq * 4;
    for (int64_t h = (int64_t)blockIdx.x * PFA_DIV_WARPS + wib; h < n_heads; h += nwarps) {
        const int64_t i0 = heads[h], i1 = (h + 1 < n_heads) ? heads[h + 1] : n_exc;
        const int64_t s = (int64_t)(keys[i0] >> 32);
        if (!pfa_div_counts<true>(b0, b1, v, masks, Wq, pop_n, k, s, lane, cnt[wib])) continue;  // pfa_divergence_kernel's site
        // D of the planes' classes, then one run of escape bytes after the other takes its equal pairs off
        for (int p = lane; p < P; p += 32) {
            const unsigned long long d = pfa_div_plane_d(cnt[wib][px[p]], cnt[wib][py[p]], pop_n, px[p], py[p]);
            if (d) atomicAdd(&tot[p], d);
            if (dsite) dsite[(int64_t)p * ns + s] = (int64_t)d;
        }
        for (int64_t r0 = i0; r0 < i1;) {
            const unsigned byte = (unsigned)((keys[r0] >> 24) & 0xffu);
            int64_t r1 = i1;
            for (int64_t base = r0 + 1; base < i1; base += 32) {  // the first key of another byte
                const int64_t idx = base + lane;
                const unsigned other = __ballot_sync(0xffffffffu, idx < i1 && ((keys[idx] >> 24) & 0xffu) != byte);
                if (other) {
                    r1 = base + __ffs(other) - 1;
                    break;
                }
            }
            for (int q = lane; q < k; q += 32) run[wib][q] = 0u;
            __syncwarp();
            for (int64_t i = r0 + lane; i < r1; i += 32) {
                const uint32_t row = (uint32_t)(keys[i] & 0xffffffull);
                for (int q = 0; q < k; ++q) {
                    const uint32_t* mq = reinterpret_cast<const uint32_t*>(masks) + (int64_t)q * Wn;
                    if ((__ldg(mq + (row >> 5)) >> (row & 31)) & 1u) atomicAdd(&run[wib][q], 1u);
                }
            }
            __syncwarp();
            for (int p = lane; p < P; p += 32) {
                const unsigned long long e = (unsigned long long)run[wib][px[p]] * run[wib][py[p]];
                if (e) {
                    atomicAdd(&tot[p], 0ull - e);  // exact modulo 2^64: the site's total stays >= 0
                    if (dsite) dsite[(int64_t)p * ns + s] -= (int64_t)e;
                }
            }
            __syncwarp();
            r0 = r1;
        }
    }
    __syncthreads();
    for (int p = threadIdx.x; p < P; p += blockDim.x)
        if (tot[p]) atomicAdd(out + p, tot[p]);
}

// dxy, d_a, F_ST of `count` entries (the operation order of the header's description of pfa_div_finalize)
__global__ void __launch_bounds__(256) pfa_div_finalize_kernel(const pfa_div_in* __restrict__ in, pfa_div_out* __restrict__ out, int count) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= count) return;
    const pfa_div_in p = in[e];
    pfa_div_out r;
    r.dxy = 0.0; r.da = 0.0; r.fst = 0.0; r.fst_is_NA = 1; r.undefined = 0;
    const int64_t nn = p.n_x * p.n_y;
    if (nn <= 0 || !(p.seqlen > 0.0)) {
        r.undefined = 1;
        out[e] = r;
        return;
    }
    double dxy = __ddiv_rn(__ddiv_rn((double)p.D, (double)nn), p.seqlen);
    if (p.jc) {  // the rule K5 applies to pi: a failing log keeps the uncorrected value
        const double x = __dsub_rn(1.0, __dmul_rn(4.0 / 3.0, dxy));
        if (x > 0.0) dxy = __dmul_rn(-0.75, log(x));
    }
    const double hw = __dmul_rn(0.5, __dadd_rn(p.pi_x, p.pi_y));
    r.dxy = dxy;
    r.da = __dsub_rn(dxy, hw);
    if (dxy != 0.0) {
        r.fst = __dsub_rn(1.0, __ddiv_rn(hw, dxy));
        r.fst_is_NA = 0;
    }
    out[e] = r;
}

static unsigned pfa_div_grid(pfa_ctx* ctx, int64_t warps) {
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((warps + PFA_DIV_WARPS - 1) / PFA_DIV_WARPS, (int64_t)ctx->sm_count * 8));
}

static int pfa_div_check(pfa_aln* a) {
    if (a->k < 2 || a->k > PFA_DIV_MAX_POPS)
        return pfa_fail(a->ctx, PFA_ERR_ARG, "divergence: needs 2 to %d populations (have %d)", PFA_DIV_MAX_POPS, a->k);
    if (a->ns > INT_MAX) return pfa_fail(a->ctx, PFA_ERR_ARG, "divergence: a shard of more than 2^31-1 sites is not supported");
    return PFA_OK;
}

static int64_t pfa_div_pairs(const pfa_aln* a) { return (int64_t)a->k * (a->k - 1) / 2; }

// d_out[P] = this shard's D_xy per pair; d_dsite (optional) = [P][ns] per-site values
static int pfa_launch_divergence(pfa_aln* a, int64_t* d_out, int64_t* d_dsite) {
    pfa_ctx* ctx = a->ctx;
    const int64_t P = pfa_div_pairs(a);
    PFA_CUDA(ctx, cudaMemsetAsync(d_out, 0, sizeof(int64_t) * (size_t)P, ctx->stream));
    if (d_dsite && a->ns > 0) PFA_CUDA(ctx, cudaMemsetAsync(d_dsite, 0, sizeof(int64_t) * (size_t)(P * a->ns), ctx->stream));
    if (a->ns == 0 || a->n == 0) return PFA_OK;
    uint8_t* flags = nullptr;
    int64_t *sites = nullptr, *d_num = nullptr;
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    cudaError_t e = pfa_dmalloc(ctx, &flags, (size_t)a->ns);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &sites, sizeof(int64_t) * (size_t)a->ns);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_num, sizeof(int64_t));
    int rc = e == cudaSuccess ? PFA_OK : pfa_fail(ctx, PFA_ERR_CUDA, "divergence: cudaMallocAsync failed: %s", cudaGetErrorString(e));
    if (!rc) rc = pfa_launch_var_flags(a, flags);
    cub::CountingInputIterator<int64_t> idx(0);
    if (!rc) {
        e = cub::DeviceSelect::Flagged(nullptr, tmp_bytes, idx, flags, sites, d_num, (int)a->ns, ctx->stream);
        if (e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
        if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(tmp, tmp_bytes, idx, flags, sites, d_num, (int)a->ns, ctx->stream);
        ctx->launches++;
        if (e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "divergence: site list failed: %s", cudaGetErrorString(e));
    }
    unsigned long long* out = reinterpret_cast<unsigned long long*>(d_out);
    const uint4* masks = a->d_masks;
    if (!rc) {
        // the number of listed sites stays on the device: the grid covers every site, warps beyond the list exit at once
        const unsigned grid = pfa_div_grid(ctx, a->ns);
        if (a->has_invalid)
            pfa_divergence_kernel<true><<<grid, 256, 0, ctx->stream>>>(a->b0, a->b1, a->v, masks, a->Wq, a->d_pop_n, a->k, sites, d_num, a->ns, out, d_dsite);
        else
            pfa_divergence_kernel<false><<<grid, 256, 0, ctx->stream>>>(a->b0, a->b1, a->v, masks, a->Wq, a->d_pop_n, a->k, sites, d_num, a->ns, out, d_dsite);
        ctx->launches++;
        e = cudaGetLastError();
        if (e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "divergence: kernel launch failed: %s", cudaGetErrorString(e));
    }
    if (!rc && a->n_exc_sites > 0) {
        pfa_divergence_escape_kernel<<<pfa_div_grid(ctx, a->n_exc_sites), 256, 0, ctx->stream>>>(
            a->b0, a->b1, a->v, masks, a->Wq, a->d_pop_n, a->k, a->exc_keys, a->n_exc, a->exc_heads, a->n_exc_sites, a->ns, out, d_dsite);
        ctx->launches++;
        e = cudaGetLastError();
        if (e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "divergence: escape kernel launch failed: %s", cudaGetErrorString(e));
    }
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, d_num);
    pfa_dfree(ctx, sites);
    pfa_dfree(ctx, flags);
    return rc;
}

static int pfa_launch_div_finalize(pfa_ctx* ctx, const pfa_div_in* d_in, pfa_div_out* d_out, int count) {
    if (count <= 0) return PFA_OK;
    pfa_div_finalize_kernel<<<(count + 255) / 256, 256, 0, ctx->stream>>>(d_in, d_out, count);
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}

extern "C" {

int pfa_divergence_device(pfa_aln* a, int64_t* d_out) {
    if (!a || !d_out) return PFA_ERR_ARG;
    if (int rc = pfa_div_check(a)) return rc;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_divergence(a, d_out, nullptr);
}

int pfa_divergence_windows_device(pfa_aln* a, int64_t window, int64_t step, int64_t* d_counts) {
    if (!a) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    if (window < 1 || step < 1) return pfa_fail(ctx, PFA_ERR_ARG, "divergence windows: window and step must be >= 1 (got %lld, %lld)", (long long)window, (long long)step);
    if (int rc = pfa_div_check(a)) return rc;
    if (pfa_window_count(a->L_total, window, step) == 0) return PFA_OK;
    if (!d_counts) return pfa_fail(ctx, PFA_ERR_ARG, "divergence windows: null output");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t P = pfa_div_pairs(a);
    int64_t *d_tot = nullptr, *d_dsite = nullptr;
    const size_t dbytes = sizeof(int64_t) * (size_t)std::max<int64_t>(P * a->ns, 1);
    cudaError_t e = pfa_dmalloc(ctx, &d_tot, sizeof(int64_t) * (size_t)P);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_dsite, dbytes);
    int rc = e == cudaSuccess ? PFA_OK
                              : pfa_fail(ctx, PFA_ERR_CUDA, "divergence windows: %zu bytes of per-site values for %lld pairs x %lld sites: %s", dbytes,
                                         (long long)P, (long long)a->ns, cudaGetErrorString(e));
    if (!rc) rc = pfa_launch_divergence(a, d_tot, d_dsite);
    if (!rc) rc = pfa_launch_row_windows(a, (int)P, d_dsite, window, step, d_counts);
    pfa_dfree(ctx, d_dsite);
    pfa_dfree(ctx, d_tot);
    return rc;
}

int pfa_div_finalize(pfa_ctx* ctx, const pfa_div_in* in, pfa_div_out* out, int count) {
    if (!ctx) return PFA_ERR_ARG;
    if (count <= 0) return PFA_OK;
    if (!in || !out) return pfa_fail(ctx, PFA_ERR_ARG, "pfa_div_finalize: null buffer");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    pfa_div_in* d_in = nullptr;
    pfa_div_out* d_out = nullptr;
    cudaError_t e = pfa_dmalloc(ctx, &d_in, sizeof(pfa_div_in) * (size_t)count);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_out, sizeof(pfa_div_out) * (size_t)count);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_in, in, sizeof(pfa_div_in) * (size_t)count, cudaMemcpyHostToDevice, ctx->stream);
    int rc = e == cudaSuccess ? PFA_OK : pfa_fail(ctx, PFA_ERR_CUDA, "pfa_div_finalize: %s", cudaGetErrorString(e));
    if (!rc) rc = pfa_launch_div_finalize(ctx, d_in, d_out, count);
    if (!rc) {
        e = cudaMemcpyAsync(out, d_out, sizeof(pfa_div_out) * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "pfa_div_finalize: result copy failed: %s", cudaGetErrorString(e));
    }
    pfa_dfree(ctx, d_out);
    pfa_dfree(ctx, d_in);
    return rc;
}

}  // extern "C"
