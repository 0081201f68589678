// K3: pairwise mismatch counts d_ij = #columns whose characters differ between rows i and j.
//
// Replaces the reference's (dead) nucleotide_diversity3 (PolyFastA.py:468-480): sum_{i<j} d_ij / C(n,2); the
// identity sum_{i<j} d_ij = H/2 ties it to the site scan.  Integer work on the INT pipe -- XOR / OR / POPC over
// packed words -- not tensor cores.
//
//  0. pfa_var_flags_kernel marks the sites at which at least two rows differ (one memory-bound pass over the planes); only
//     those can contribute to any d_ij -- the reference, too, runs over the variable columns only (:469) -- and they are
//     a few per cent of a real alignment, so the K dimension of step 2 shrinks by that factor.
//  1. pfa_rowmajor_kernel transposes the marked sites of the site-major planes into row-major bit-planes over SITES
//     ([plane][row][word], 32 sites per word) with warp ballots.  Steps 0 and 1 run once per alignment (pfa_rowmajor_ensure):
//     the planes and the list of marked sites stay with the alignment, and the haplotype classes (pfa_haplotypes.cu) reuse them.
//  2. pfa_pairwise_kernel: one 64x64 tile of row pairs per CTA, 4x4 pairs per thread; the K dimension (site words)
//     is staged through shared memory in [plane][word][row] order so that a thread fetches its four rows with one
//     128-bit shared load; per word and pair: mismatch = (a0^b0)|(a1^b1)|(av^bv), POPC, add.
//  3. rows that both show the escape class compare equal in the planes; pfa_pairwise_escape_kernel adds the pairs
//     whose escape BYTES differ from the sorted exception list.
//  4. pfa_pairwise_popsum_kernel reduces the upper triangle per population.
// A pure-ACGT shard (no validity plane needed) runs the two-plane instantiations: a third fewer logic ops and shared-memory
// traffic in step 2.  When the caller wants only the sums, the n x n matrix is never written: every tile folds its pairs
// into the per-population sums in registers (pfa_pairwise_kernel<NP, false>).
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "pfa_common.cuh"

#define PW_TILE 64
#define PW_KC 16
#define PW_LD (PW_TILE + 4)  // row pitch of the staged tiles: the transposing stores hit 2 banks twice instead of 1 bank 16 times

// one warp per site: does any plane show both a 0 and a 1 among the n rows?  (rows beyond n are padding)
template <int NP>
__global__ void __launch_bounds__(256) pfa_var_flags_kernel(const uint4* __restrict__ b0, const uint4* __restrict__ b1,
                                                            const uint4* __restrict__ v, int64_t ns, int Wq, int64_t n,
                                                            uint8_t* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int64_t site = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (site >= ns) return;
    uint32_t o[3] = {0, 0, 0}, z[3] = {0, 0, 0};
    const uint4* planes[3] = {b0, b1, v};
    for (int j = lane; j < Wq; j += 32) {
        uint32_t m[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int64_t lo = ((int64_t)j * 4 + w) * 32;
            m[w] = lo + 32 <= n ? 0xffffffffu : (lo >= n ? 0u : ((1u << (n - lo)) - 1u));
        }
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const uint4 x = __ldg(planes[p] + site * Wq + j);
            o[p] |= (x.x & m[0]) | (x.y & m[1]) | (x.z & m[2]) | (x.w & m[3]);
            z[p] |= (~x.x & m[0]) | (~x.y & m[1]) | (~x.z & m[2]) | (~x.w & m[3]);
        }
    }
    unsigned both = 0;
#pragma unroll
    for (int p = 0; p < NP; ++p) {
        const unsigned any_o = __any_sync(0xffffffffu, o[p] != 0), any_z = __any_sync(0xffffffffu, z[p] != 0);
        both |= (any_o && any_z) ? 1u : 0u;
    }
    if (lane == 0) flags[site] = (uint8_t)both;
}

// sites[i]: the i-th marked site; word sw of the row-major planes holds marked sites 32*sw .. 32*sw+31
template <int NP>
__global__ void __launch_bounds__(256) pfa_rowmajor_kernel(const uint32_t* __restrict__ b0, const uint32_t* __restrict__ b1,
                                                           const uint32_t* __restrict__ v, const int64_t* __restrict__ sites,
                                                           int64_t nsel, int Wn, int64_t npad, int64_t Wl,
                                                           uint32_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t sw = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // word over marked sites
    const int64_t w = blockIdx.y;                                                      // word over rows
    if (sw * 32 >= nsel) return;
    const int64_t idx = sw * 32 + lane;
    const int64_t site = idx < nsel ? sites[idx] : -1;
    const uint32_t* planes[3] = {b0, b1, v};
#pragma unroll
    for (int p = 0; p < NP; ++p) {
        const uint32_t x = site >= 0 ? __ldg(planes[p] + site * Wn + w) : 0u;
        uint32_t mine = 0;
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const uint32_t word = __ballot_sync(0xffffffffu, (x >> r) & 1u);
            if (lane == r) mine = word;
        }
        const int64_t row = w * 32 + lane;
        out[((int64_t)p * npad + row) * Wl + sw] = mine;
    }
}

// NP: planes compared (2 for a pure-ACGT shard).  WANT_D: write the n x n matrix; otherwise fold the tile's pairs (i < j, both
// rows in the population) into the per-population sums -- masks: [k][Wn] row masks, out: [k]
template <int NP, bool WANT_D>
__global__ void __launch_bounds__(256) pfa_pairwise_kernel(const uint32_t* __restrict__ rm, int64_t npad, int64_t Wl, int64_t n,
                                                           int32_t* __restrict__ D, const uint32_t* __restrict__ masks, int Wn, int k,
                                                           int64_t* __restrict__ out) {
    // upper-triangular tile index -> (bi, bj), bj >= bi
    const int nt = (int)(npad / PW_TILE);
    int bi = 0, rem = blockIdx.x;
    while (rem >= nt - bi) { rem -= nt - bi; ++bi; }
    const int bj = bi + rem;
    __shared__ __align__(16) uint32_t As[NP][PW_KC][PW_LD];
    __shared__ __align__(16) uint32_t Bs[NP][PW_KC][PW_LD];
    const int tj = threadIdx.x & 15, ti = threadIdx.x >> 4;
    int acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0;
    for (int64_t k0 = 0; k0 < Wl; k0 += PW_KC) {
        // stage 64 rows x PW_KC words x NP planes of both tiles; consecutive threads read consecutive words of a row
        for (int idx = threadIdx.x; idx < NP * PW_TILE * PW_KC; idx += 256) {
            const int kw = idx % PW_KC, r = (idx / PW_KC) % PW_TILE, p = idx / (PW_KC * PW_TILE);
            const int64_t kk = k0 + kw;
            uint32_t a = 0, b = 0;
            if (kk < Wl) {
                a = __ldg(rm + ((int64_t)p * npad + (int64_t)bi * PW_TILE + r) * Wl + kk);
                b = __ldg(rm + ((int64_t)p * npad + (int64_t)bj * PW_TILE + r) * Wl + kk);
            }
            As[p][kw][r] = a;
            Bs[p][kw][r] = b;
        }
        __syncthreads();
#pragma unroll 4
        for (int kw = 0; kw < PW_KC; ++kw) {
            const uint4 a0 = *reinterpret_cast<const uint4*>(&As[0][kw][ti * 4]);
            const uint4 a1 = *reinterpret_cast<const uint4*>(&As[1][kw][ti * 4]);
            const uint4 c0 = *reinterpret_cast<const uint4*>(&Bs[0][kw][tj * 4]);
            const uint4 c1 = *reinterpret_cast<const uint4*>(&Bs[1][kw][tj * 4]);
            uint4 av = make_uint4(0, 0, 0, 0), cv = make_uint4(0, 0, 0, 0);
            if (NP == 3) {
                av = *reinterpret_cast<const uint4*>(&As[NP - 1][kw][ti * 4]);
                cv = *reinterpret_cast<const uint4*>(&Bs[NP - 1][kw][tj * 4]);
            }
            const uint32_t A0[4] = {a0.x, a0.y, a0.z, a0.w}, A1[4] = {a1.x, a1.y, a1.z, a1.w}, AV[4] = {av.x, av.y, av.z, av.w};
            const uint32_t B0[4] = {c0.x, c0.y, c0.z, c0.w}, B1[4] = {c1.x, c1.y, c1.z, c1.w}, BV[4] = {cv.x, cv.y, cv.z, cv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t d = (A0[i] ^ B0[j]) | (A1[i] ^ B1[j]);
                    if (NP == 3) d |= AV[i] ^ BV[j];
                    acc[i][j] += __popc(d);
                }
        }
        __syncthreads();
    }
    if (WANT_D) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int64_t r = (int64_t)bi * PW_TILE + ti * 4 + i, c = (int64_t)bj * PW_TILE + tj * 4 + j;
                if (r < n && c < n) {
                    D[r * n + c] = acc[i][j];
                    D[c * n + r] = acc[i][j];
                }
            }
        return;
    }
    // sums only: pairs i < j with both rows in the population (rows beyond n are in no mask)
    __shared__ unsigned long long red[8];
    const int r0 = bi * PW_TILE + ti * 4, c0 = bj * PW_TILE + tj * 4;  // multiples of 4: the four mask bits sit in one word
    for (int q = 0; q < k; ++q) {
        const uint32_t* mq = masks + (int64_t)q * Wn;
        const unsigned rb = (mq[r0 >> 5] >> (r0 & 31)) & 0xfu, cb = (mq[c0 >> 5] >> (c0 & 31)) & 0xfu;
        unsigned long long s = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (((rb >> i) & 1u) && ((cb >> j) & 1u) && r0 + i < c0 + j) s += (unsigned long long)acc[i][j];
        for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long t = 0;
            for (int w = 0; w < 8; ++w) t += red[w];
            if (t) atomicAdd(reinterpret_cast<unsigned long long*>(out + q), t);
        }
        __syncthreads();
    }
}

// pairs of rows that both carry an escape symbol at a site but different bytes: one more mismatch each
// D != nullptr: into the matrix; else straight into the per-population sums (masks: [k][Wn])
__global__ void __launch_bounds__(256) pfa_pairwise_escape_kernel(const unsigned long long* __restrict__ keys, int64_t n_exc,
                                                                  const int64_t* __restrict__ heads, int64_t n_heads, int64_t n,
                                                                  int32_t* __restrict__ D, const uint32_t* __restrict__ masks, int Wn, int k,
                                                                  int64_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t h = wid; h < n_heads; h += nwarps) {
        const int64_t i0 = heads[h], i1 = (h + 1 < n_heads) ? heads[h + 1] : n_exc;
        const int64_t m = i1 - i0;
        for (int64_t p = lane; p < m * m; p += 32) {
            const int64_t x = p / m, y = p % m;
            if (x >= y) continue;
            const unsigned long long kx = keys[i0 + x], ky = keys[i0 + y];
            if (((kx >> 24) & 0xff) == ((ky >> 24) & 0xff)) continue;
            const int64_t rx = (int64_t)(kx & 0xffffff), ry = (int64_t)(ky & 0xffffff);
            if (D) {
                atomicAdd(&D[rx * n + ry], 1);
                atomicAdd(&D[ry * n + rx], 1);
            } else {
                for (int q = 0; q < k; ++q) {
                    const uint32_t* mq = masks + (int64_t)q * Wn;
                    if (((mq[rx >> 5] >> (rx & 31)) & 1u) && ((mq[ry >> 5] >> (ry & 31)) & 1u))
                        atomicAdd(reinterpret_cast<unsigned long long*>(out + q), 1ull);
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) pfa_pairwise_popsum_kernel(const int32_t* __restrict__ D, int64_t n, const uint32_t* __restrict__ masks,
                                                                  int Wn, int k, int64_t* __restrict__ out) {
    const int64_t i = blockIdx.x;
    __shared__ unsigned long long red[8];
    for (int q = 0; q < k; ++q) {
        const uint32_t* mq = masks + (int64_t)q * Wn;
        if (!((mq[i >> 5] >> (i & 31)) & 1u)) continue;  // block-uniform
        unsigned long long s = 0;
        for (int64_t j = i + 1 + threadIdx.x; j < n; j += blockDim.x)
            if ((mq[j >> 5] >> (j & 31)) & 1u) s += (unsigned long long)D[i * n + j];
        for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long t = 0;
            for (int w = 0; w < 8; ++w) t += red[w];
            if (t) atomicAdd(reinterpret_cast<unsigned long long*>(out + q), t);
        }
        __syncthreads();
    }
}

// step 0 alone, for the divergence scan (pfa_divergence.cu): flags[s] = 1 where two rows differ in the planes; the two-plane
// instantiation for a pure-ACGT shard, as below
int pfa_launch_var_flags(pfa_aln* a, uint8_t* flags) {
    pfa_ctx* ctx = a->ctx;
    if (a->ns == 0) return PFA_OK;
    const unsigned g = (unsigned)((a->ns + 7) / 8);
    if (a->has_invalid) pfa_var_flags_kernel<3><<<g, 256, 0, ctx->stream>>>(a->b0, a->b1, a->v, a->ns, a->Wq, a->n, flags);
    else pfa_var_flags_kernel<2><<<g, 256, 0, ctx->stream>>>(a->b0, a->b1, a->v, a->ns, a->Wq, a->n, flags);
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}

// steps 0 and 1, cached with the alignment: the row-major planes of the marked sites and the sorted list of those sites (a
// window [s, e) of this shard is the bit range [lower_bound(s), lower_bound(e)) of the row-major words).  Rebuilt when the
// number of planes changes (pfa_aln_force_validity).
cudaError_t pfa_rowmajor_ensure(pfa_aln* a) {
    pfa_ctx* ctx = a->ctx;
    const int64_t n = a->n;
    const bool three = a->has_invalid != 0;  // the validity plane takes part only when a row shows a symbol outside ACGT
    const int np = three ? 3 : 2;
    if (a->ns == 0 || n == 0 || (a->rowmajor && a->rowmajor_planes == np)) return cudaSuccess;
    pfa_dfree(ctx, a->rowmajor);
    pfa_dfree(ctx, a->rowmajor_sites);
    a->rowmajor = nullptr;
    a->rowmajor_sites = nullptr;
    a->rowmajor_nsel = 0;
    const int Wn = a->Wq * 4;
    const int64_t npad = (int64_t)a->Wq * 128;
    // mark the sites at which two rows differ, list them, transpose only those
    uint8_t* flags = nullptr;
    int64_t *sites = nullptr, *d_num = nullptr;
    void* tmp = nullptr;
    size_t tmp_bytes = 0;
    int64_t nsel = 0;
    cudaError_t e = pfa_dmalloc(ctx, &flags, (size_t)a->ns);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &sites, sizeof(int64_t) * (size_t)a->ns);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_num, sizeof(int64_t));
    if (e == cudaSuccess) {
        const unsigned g = (unsigned)((a->ns + 7) / 8);
        if (three) pfa_var_flags_kernel<3><<<g, 256, 0, ctx->stream>>>(a->b0, a->b1, a->v, a->ns, a->Wq, n, flags);
        else pfa_var_flags_kernel<2><<<g, 256, 0, ctx->stream>>>(a->b0, a->b1, a->v, a->ns, a->Wq, n, flags);
        ctx->launches++;
        e = cudaGetLastError();
    }
    cub::CountingInputIterator<int64_t> idx(0);
    if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(nullptr, tmp_bytes, idx, flags, sites, d_num, (int)a->ns, ctx->stream);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &tmp, tmp_bytes);
    if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(tmp, tmp_bytes, idx, flags, sites, d_num, (int)a->ns, ctx->stream);
    ctx->launches += 2;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&nsel, d_num, sizeof nsel, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) {
        a->Wl = pfa_round_up(std::max<int64_t>((nsel + 31) / 32, 1), 4);
        a->rowmajor_planes = np;
        e = pfa_dmalloc(ctx, &a->rowmajor, sizeof(uint32_t) * (size_t)(np * npad * a->Wl));
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(a->rowmajor, 0, sizeof(uint32_t) * (size_t)(np * npad * a->Wl), ctx->stream);
    if (e == cudaSuccess && nsel > 0) {
        const int64_t sw = (nsel + 31) / 32;
        dim3 grid((unsigned)((sw + 7) / 8), (unsigned)Wn);
        if (three)
            pfa_rowmajor_kernel<3><<<grid, 256, 0, ctx->stream>>>((const uint32_t*)a->b0, (const uint32_t*)a->b1, (const uint32_t*)a->v, sites, nsel,
                                                                  Wn, npad, a->Wl, a->rowmajor);
        else
            pfa_rowmajor_kernel<2><<<grid, 256, 0, ctx->stream>>>((const uint32_t*)a->b0, (const uint32_t*)a->b1, (const uint32_t*)a->v, sites, nsel,
                                                                  Wn, npad, a->Wl, a->rowmajor);
        ctx->launches++;
        e = cudaGetLastError();
    }
    pfa_dfree(ctx, tmp);
    pfa_dfree(ctx, flags);
    pfa_dfree(ctx, d_num);
    if (e == cudaSuccess) {
        a->rowmajor_sites = sites;  // the first nsel entries: the marked sites in ascending order
        a->rowmajor_nsel = nsel;
    } else {
        pfa_dfree(ctx, sites);
        pfa_dfree(ctx, a->rowmajor);
        a->rowmajor = nullptr;
        a->rowmajor_planes = 0;
    }
    return e;
}

int pfa_launch_pairwise(pfa_aln* a, int64_t* d_out, int32_t* d_matrix) {
    pfa_ctx* ctx = a->ctx;
    PFA_CUDA(ctx, cudaMemsetAsync(d_out, 0, sizeof(int64_t) * (size_t)a->k, ctx->stream));
    const int64_t n = a->n;
    if (n == 0) return PFA_OK;
    if (a->ns > 0x7fffffffll) return pfa_fail(ctx, PFA_ERR_ARG, "pairwise: a shard of more than 2^31-1 sites is not supported");
    int32_t* D = d_matrix;  // nullptr: sums only, the matrix is never materialised
    const int Wn = a->Wq * 4;
    const int64_t npad = (int64_t)a->Wq * 128;
    const bool three = a->has_invalid != 0;
    int rc = PFA_OK;
    cudaError_t e = cudaSuccess;
    if (D) e = cudaMemsetAsync(D, 0, sizeof(int32_t) * (size_t)(n * n), ctx->stream);
    if (e == cudaSuccess && a->ns > 0) {
        e = pfa_rowmajor_ensure(a);
        if (e == cudaSuccess) {
            const int64_t nt = npad / PW_TILE;
            const unsigned grid = (unsigned)(nt * (nt + 1) / 2);
            const uint32_t* masks = (const uint32_t*)a->d_masks;
#define PFA_PW(NP_, WD_) pfa_pairwise_kernel<NP_, WD_><<<grid, 256, 0, ctx->stream>>>(a->rowmajor, npad, a->Wl, n, D, masks, Wn, a->k, d_out)
            if (three && D) PFA_PW(3, true);
            else if (three) PFA_PW(3, false);
            else if (D) PFA_PW(2, true);
            else PFA_PW(2, false);
#undef PFA_PW
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess && a->n_exc_sites > 0) {
            int64_t eb = std::min<int64_t>((a->n_exc_sites + 7) / 8, (int64_t)ctx->sm_count * 8);
            pfa_pairwise_escape_kernel<<<(unsigned)eb, 256, 0, ctx->stream>>>(a->exc_keys, a->n_exc, a->exc_heads, a->n_exc_sites, n, D,
                                                                           (const uint32_t*)a->d_masks, Wn, a->k, d_out);
            ctx->launches++;
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess && D) {
        pfa_pairwise_popsum_kernel<<<(unsigned)n, 256, 0, ctx->stream>>>(D, n, (const uint32_t*)a->d_masks, Wn, a->k, d_out);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "pairwise failed: %s", cudaGetErrorString(e));
    return rc;
}
