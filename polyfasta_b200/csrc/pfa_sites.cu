// K2: per-site allele counting over the packed alignment.
//
// Replaces getvarsites (PolyFastA.py:252-261) and the column sums inside nucleotide_diversity (:485-492),
// wattersons_theta (:494-497) and getsfs (:274-282): one pass over the planes yields, for every population at
// once, S = #columns with > 1 distinct character, H = sum_cols (n^2 - sum_a c_a^2) and the folded SFS.
//
// A warp owns one site; its lanes stride over the Wq 128-bit chunks of the site record.
// Pass 1 (every site, 2 or 3 coalesced 128-bit loads per chunk, logic ops only) decides whether all rows
// of the union of the populations carry the same symbol.  Monomorphic sites -- the overwhelming majority of
// a real alignment -- end there.  Pass 2 (variable sites only; re-reads the record from L1/L2) counts the
// symbol classes per population with popcounts and warp reductions.  Sites holding "escape" symbols (IUPAC
// codes etc., which are distinct alleles in the reference) are finished by pfa_escape_sites_kernel from the
// sorted exception list.
#include <cstdio>
#include <cstdlib>

#include "pfa_sites.cuh"

template <bool HAS_V>
__global__ void __launch_bounds__(PFA_SITE_THREADS) pfa_site_scan_kernel(const PfaSiteArgs a) {
    extern __shared__ unsigned long long smem[];
    if (a.x.world && blockIdx.x == 0 && threadIdx.x == 0) a.x.stamps[5] = pfa_globaltimer();
    unsigned long long* sm_SH = smem;                                       // [2k]
    unsigned int* sm_sfs = reinterpret_cast<unsigned int*>(smem + 2 * a.k);  // [sfs_bins] when a.sfs_in_smem
    const int nsm = 2 * a.k;
    for (int i = threadIdx.x; i < nsm; i += blockDim.x) sm_SH[i] = 0ull;
    if (a.sfs_in_smem)
        for (int i = threadIdx.x; i < a.sfs_bins; i += blockDim.x) sm_sfs[i] = 0u;
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const int64_t nwarps = (int64_t)gridDim.x * blockDim.x / 32;
    const int Wq = a.Wq;

    for (int64_t s = wid; s < a.ns; s += nwarps) {
        const uint4* p0 = a.b0 + s * Wq;
        const uint4* p1 = a.b1 + s * Wq;
        const uint4* pv = a.v + s * Wq;
        // ---- pass 1: is the column monomorphic over the union of the populations? ----
        uint32_t o0 = 0, z0 = 0, o1 = 0, z1 = 0, ov = 0, zv = 0;
#pragma unroll 2
        for (int j = lane; j < Wq; j += 32) {
            const uint4 m = __ldg(a.umask + j);
            const uint4 x0 = pfa_ld_stream(p0 + j);
            const uint4 x1 = pfa_ld_stream(p1 + j);
            o0 |= (x0.x & m.x) | (x0.y & m.y) | (x0.z & m.z) | (x0.w & m.w);
            z0 |= (~x0.x & m.x) | (~x0.y & m.y) | (~x0.z & m.z) | (~x0.w & m.w);
            o1 |= (x1.x & m.x) | (x1.y & m.y) | (x1.z & m.z) | (x1.w & m.w);
            z1 |= (~x1.x & m.x) | (~x1.y & m.y) | (~x1.z & m.z) | (~x1.w & m.w);
            if (HAS_V) {
                const uint4 xv = pfa_ld_stream(pv + j);
                ov |= (xv.x & m.x) | (xv.y & m.y) | (xv.z & m.z) | (xv.w & m.w);
                zv |= (~xv.x & m.x) | (~xv.y & m.y) | (~xv.z & m.z) | (~xv.w & m.w);
            } else {
                ov |= m.x | m.y | m.z | m.w;
            }
        }
        unsigned f = (o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (ov ? 16u : 0u) | (zv ? 32u : 0u);
        f = __reduce_or_sync(0xffffffffu, f);
        const bool mono = ((f & 3u) != 3u) && ((f & 12u) != 12u) && ((f & 48u) != 48u);
        const bool all_escape = (f & 1u) && (f & 4u) && !(f & 16u);  // every row shows the escape class
        if (mono && !all_escape) {
            if (a.isvar && lane == 0)
                for (int q = 0; q < a.k; ++q) a.isvar[(int64_t)q * a.ns + s] = 0;
            continue;
        }
        // ---- pass 2: class counts per population ----
        for (int q = 0; q < a.k; ++q) {
            uint32_t c[PFA_NCLASS];
            pfa_class_counts<HAS_V>(p0, p1, pv, a.masks + (int64_t)q * Wq, Wq, lane, c);
            if (lane != 0) continue;
            const int64_t nq = a.pop_n[q];
            PfaSiteResult r = pfa_site_result(c, nq, 0u, 0ull);
            if (r.has_escape) continue;  // finished by pfa_escape_sites_kernel
            if (a.isvar) a.isvar[(int64_t)q * a.ns + s] = (uint8_t)r.isvar;
            if (r.isvar) {
                if (a.hsite) a.hsite[(int64_t)q * a.ns + s] = (int64_t)r.h;
                atomicAdd(&sm_SH[2 * q], 1ull);
                atomicAdd(&sm_SH[2 * q + 1], r.h);
                if (r.sfs_bin >= 0) {
                    if (a.sfs_in_smem) atomicAdd(&sm_sfs[a.sfs_off[q] + r.sfs_bin], 1u);
                    else atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + r.sfs_bin), 1ull);
                }
            }
        }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < a.k; q += blockDim.x) {
        if (sm_SH[2 * q]) {
            atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q]), sm_SH[2 * q]);
            atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 1), sm_SH[2 * q + 1]);
        }
    }
    if (a.sfs_in_smem) {
        for (int q = 0; q < a.k; ++q) {
            const int nb = (int)(a.pop_n[q] / 2);
            for (int i = threadIdx.x; i < nb; i += blockDim.x) {
                const unsigned int cnt = sm_sfs[a.sfs_off[q] + i];
                if (cnt) atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + i), (unsigned long long)cnt);
            }
        }
    }
    if (a.x.world) pfa_xchg_epilogue(a.x);
}

// passes 1 and 2 of one site whose record chunks are already in registers (x0, x1, xv: the lane's ITER chunks of each plane;
// um: its slice of the union mask).  Shared by the register-resident kernel (chunks loaded from global memory) and the
// TMA kernel (chunks read from the warp's shared-memory ring).
// pass 1 of one site whose chunks are in registers: the six presence flags, OR-reduced over the group.
// VALID_ONLY (with HAS_V): the flags of the two base planes look at the VALID rows only, so that "every valid row shows the same
// base" can be told apart from real base variation (the gap-only fast path of the whole-warp second pass).
template <int LPS, int ITER, bool HAS_V, bool VALID_ONLY = false>
__device__ __forceinline__ unsigned pfa_site_pass1(const uint4 (&x0)[ITER], const uint4 (&x1)[ITER], const uint4 (&xv)[ITER],
                                                   const uint4 (&um)[ITER], unsigned gmask) {
    uint32_t o0 = 0, z0 = 0, o1 = 0, z1 = 0, ov = 0, zv = 0;
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        uint4 m = um[i];
        ov |= (xv[i].x & m.x) | (xv[i].y & m.y) | (xv[i].z & m.z) | (xv[i].w & m.w);
        if (HAS_V) zv |= (~xv[i].x & m.x) | (~xv[i].y & m.y) | (~xv[i].z & m.z) | (~xv[i].w & m.w);
        if (HAS_V && VALID_ONLY) m = make_uint4(m.x & xv[i].x, m.y & xv[i].y, m.z & xv[i].z, m.w & xv[i].w);
        o0 |= (x0[i].x & m.x) | (x0[i].y & m.y) | (x0[i].z & m.z) | (x0[i].w & m.w);
        z0 |= (~x0[i].x & m.x) | (~x0[i].y & m.y) | (~x0[i].z & m.z) | (~x0[i].w & m.w);
        o1 |= (x1[i].x & m.x) | (x1[i].y & m.y) | (x1[i].z & m.z) | (x1[i].w & m.w);
        z1 |= (~x1[i].x & m.x) | (~x1[i].y & m.y) | (~x1[i].z & m.z) | (~x1[i].w & m.w);
    }
    const unsigned f = (o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (ov ? 16u : 0u) | (zv ? 32u : 0u);
    return pfa_group_or<LPS>(f, gmask);
}

// pass 1 of a site of a block that carries validity pieces: mv = the lane's slice of "row belongs to the union AND is valid"
// (um where the cell is not flagged).  Bits 0-3: the base planes over the valid rows, bit 5: some row is not valid.
template <int LPS, int ITER>
__device__ __forceinline__ unsigned pfa_site_pass1_valid(const uint4 (&x0)[ITER], const uint4 (&x1)[ITER], const uint4 (&mv)[ITER],
                                                         const uint4 (&um)[ITER], unsigned gmask) {
    uint32_t o0 = 0, z0 = 0, o1 = 0, z1 = 0, zv = 0;
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        const uint4 m = mv[i];
        zv |= (um[i].x ^ m.x) | (um[i].y ^ m.y) | (um[i].z ^ m.z) | (um[i].w ^ m.w);
        o0 |= (x0[i].x & m.x) | (x0[i].y & m.y) | (x0[i].z & m.z) | (x0[i].w & m.w);
        z0 |= (~x0[i].x & m.x) | (~x0[i].y & m.y) | (~x0[i].z & m.z) | (~x0[i].w & m.w);
        o1 |= (x1[i].x & m.x) | (x1[i].y & m.y) | (x1[i].z & m.z) | (x1[i].w & m.w);
        z1 |= (~x1[i].x & m.x) | (~x1[i].y & m.y) | (~x1[i].z & m.z) | (~x1[i].w & m.w);
    }
    const unsigned f = (o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (zv ? 32u : 0u);
    return pfa_group_or<LPS>(f, gmask);
}

// pass 2 of one site on registers, given the flags of pass 1 (f, OR-reduced over the group): shared by the register-resident
// kernel and the TMA kernel's per-group path
template <int LPS, int ITER, bool HAS_V, bool MULTI>
__device__ __forceinline__ void pfa_site_finish_regs(const PfaSiteArgs& a, int64_t s, unsigned f, const uint4 (&x0)[ITER], const uint4 (&x1)[ITER],
                                                     const uint4 (&xv)[ITER], const uint4 (&um)[ITER], int sub, unsigned gmask, int Wq,
                                                     unsigned long long* sm_SH, unsigned int* sm_sfs) {
    constexpr bool one_pop = !MULTI;  // one population: its mask is the union mask, lane 0 finishes the site at once
    const bool mono = pfa_flags_mono(f), all_escape = pfa_flags_all_escape(f);
    if (mono && !all_escape) {
        if (a.isvar && sub == 0)
            for (int q = 0; q < a.k; ++q) a.isvar[(int64_t)q * a.ns + s] = 0;
        return;
    }
    // ---- pass 2 on registers ----
    // The popcounts of a population run on all lanes of the group and every lane ends up with the group's sums; what
    // follows per population (distinct symbols, H, SFS bin, accumulator updates) is scalar work.  Lane q of the group
    // keeps population q's sums and the scalar parts of all populations run side by side after the loop instead of one
    // after the other on lane 0 (with more populations than lanes a lane finishes its previous one first).
    uint32_t mine[PFA_NCLASS];
    int myq = -1;
    auto finish = [&](int q, const uint32_t (&c)[PFA_NCLASS]) {
        const int64_t nq = a.pop_n[q];
        PfaSiteResult r = pfa_site_result(c, nq, 0u, 0ull);
        if (r.has_escape) return;
        if (a.isvar) a.isvar[(int64_t)q * a.ns + s] = (uint8_t)r.isvar;
        if (r.isvar) {
            if (a.hsite) a.hsite[(int64_t)q * a.ns + s] = (int64_t)r.h;
            atomicAdd(&sm_SH[2 * q], 1ull);
            atomicAdd(&sm_SH[2 * q + 1], r.h);
            if (r.sfs_bin >= 0) {
                if (a.sfs_in_smem) atomicAdd(&sm_sfs[a.sfs_off[q] + r.sfs_bin], 1u);
                else atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + r.sfs_bin), 1ull);
            }
        }
    };
    for (int q = 0; q < a.k; ++q) {
        uint32_t c[PFA_NCLASS];
#pragma unroll
        for (int i = 0; i < PFA_NCLASS; ++i) c[i] = 0;
        const uint4* mq = a.masks + (int64_t)q * Wq;
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            const int j = sub + LPS * i;
            uint4 m4 = um[i];
            if (!one_pop) m4 = j < Wq ? __ldg(mq + j) : make_uint4(0, 0, 0, 0);
            const uint32_t m[4] = {m4.x, m4.y, m4.z, m4.w}, w0[4] = {x0[i].x, x0[i].y, x0[i].z, x0[i].w},
                           w1[4] = {x1[i].x, x1[i].y, x1[i].z, x1[i].w}, wv[4] = {xv[i].x, xv[i].y, xv[i].z, xv[i].w};
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const uint32_t vm = HAS_V ? (wv[w] & m[w]) : m[w];
                const uint32_t hi = vm & w1[w], lo = vm & ~w1[w];
                c[PFA_C_T] += __popc(hi & w0[w]);
                c[PFA_C_G] += __popc(hi & ~w0[w]);
                c[PFA_C_C] += __popc(lo & w0[w]);
                c[PFA_C_A] += __popc(lo & ~w0[w]);
                if (HAS_V) {
                    const uint32_t im = ~wv[w] & m[w];
                    const uint32_t ihi = im & w1[w];
                    c[PFA_C_ESC] += __popc(ihi & w0[w]);
                    c[PFA_C_Q] += __popc(ihi & ~w0[w]);
                    c[PFA_C_N] += __popc(im & ~w1[w] & w0[w]);
                }
            }
        }
        if (LPS > 1) {
#pragma unroll
            for (int i = 0; i < PFA_NCLASS; ++i)
                if (HAS_V || i < 4) c[i] = pfa_group_add<LPS>(c[i], gmask);
        }
        if (one_pop) {  // the common single-population case keeps its short path: lane 0 finishes at once
            if (sub == 0) finish(0, c);
            return;
        }
        if (sub == (q & (LPS - 1))) {
            if (myq >= 0) finish(myq, mine);
#pragma unroll
            for (int i = 0; i < PFA_NCLASS; ++i) mine[i] = c[i];
            myq = q;
        }
    }
    if (myq >= 0) finish(myq, mine);
}


// passes 1 and 2 of one site whose record chunks are already in registers (x0, x1, xv: the lane's ITER chunks of each plane;
// um: its slice of the union mask)
template <int LPS, int ITER, bool HAS_V, bool MULTI>
__device__ __forceinline__ void pfa_site_process(const PfaSiteArgs& a, int64_t s, const uint4 (&x0)[ITER], const uint4 (&x1)[ITER],
                                                 const uint4 (&xv)[ITER], const uint4 (&um)[ITER], int sub, unsigned gmask, int Wq,
                                                 unsigned long long* sm_SH, unsigned int* sm_sfs) {
    const unsigned f = pfa_site_pass1<LPS, ITER, HAS_V>(x0, x1, xv, um, gmask);
    pfa_site_finish_regs<LPS, ITER, HAS_V, MULTI>(a, s, f, x0, x1, xv, um, sub, gmask, Wq, sm_SH, sm_sfs);
}

// Register-resident variant for Wq <= 5*32 chunks: every lane owns ITER fixed chunks of the site record, loads them
// once (all loads of a site are issued back to back: 2-3 * ITER independent 128-bit requests per lane), keeps its slice
// of the union mask in registers for the whole kernel, and both passes work on registers -- each byte of the planes
// crosses L2 exactly once.
template <int LPS, int ITER, bool HAS_V, bool MULTI>
__global__ void __launch_bounds__(PFA_SITE_THREADS, 2) pfa_site_scan_reg_kernel(const PfaSiteArgs a) {
    extern __shared__ unsigned long long smem[];
    if (a.x.world && blockIdx.x == 0 && threadIdx.x == 0) a.x.stamps[5] = pfa_globaltimer();
    unsigned long long* sm_SH = smem;
    unsigned int* sm_sfs = reinterpret_cast<unsigned int*>(smem + 2 * a.k);
    for (int i = threadIdx.x; i < 2 * a.k; i += blockDim.x) sm_SH[i] = 0ull;
    if (a.sfs_in_smem)
        for (int i = threadIdx.x; i < a.sfs_bins; i += blockDim.x) sm_sfs[i] = 0u;
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int sub = lane & (LPS - 1);
    const unsigned gmask = LPS == 32 ? 0xffffffffu : (((1u << LPS) - 1u) << (lane - sub));
    const int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPS;
    const int64_t ngroups = (int64_t)gridDim.x * blockDim.x / LPS;
    const int Wq = a.Wq;

    uint4 um[ITER];
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        const int j = sub + LPS * i;
        um[i] = j < Wq ? __ldg(a.umask + j) : make_uint4(0, 0, 0, 0);
    }

    for (int64_t s = gid; s < a.ns; s += ngroups) {
        const uint4* p0 = a.b0 + s * Wq;
        const uint4* p1 = a.b1 + s * Wq;
        const uint4* pv = a.v + s * Wq;
        uint4 x0[ITER], x1[ITER], xv[ITER];
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            const int j = sub + LPS * i;
            x0[i] = x1[i] = make_uint4(0, 0, 0, 0);
            xv[i] = um[i];
            if (j < Wq) {
                x0[i] = pfa_ld_stream(p0 + j);
                x1[i] = pfa_ld_stream(p1 + j);
                if (HAS_V) xv[i] = pfa_ld_stream(pv + j);
            }
        }
        pfa_site_process<LPS, ITER, HAS_V, MULTI>(a, s, x0, x1, xv, um, sub, gmask, Wq, sm_SH, sm_sfs);
    }
    __syncthreads();
    for (int q = threadIdx.x; q < a.k; q += blockDim.x) {
        if (sm_SH[2 * q]) {
            atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q]), sm_SH[2 * q]);
            atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 1), sm_SH[2 * q + 1]);
        }
    }
    if (a.sfs_in_smem) {
        for (int q = 0; q < a.k; ++q) {
            const int nb = (int)(a.pop_n[q] / 2);
            for (int i = threadIdx.x; i < nb; i += blockDim.x) {
                const unsigned int cnt = sm_sfs[a.sfs_off[q] + i];
                if (cnt) atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + i), (unsigned long long)cnt);
            }
        }
    }
    if (a.x.world) pfa_xchg_epilogue(a.x);
}

// One warp per site that holds at least one escape symbol.  For every population with an escape row at
// this site the column is counted in full: the seven packed classes from the planes plus one count per
// distinct escape byte from the exception list (sorted by site, byte, row).
__global__ void __launch_bounds__(256) pfa_escape_sites_kernel(const PfaSiteArgs a, const unsigned long long* __restrict__ keys,
                                                               int64_t n_exc, const int64_t* __restrict__ heads, int64_t n_heads) {
    __shared__ unsigned int hist[8][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t h = wid; h < n_heads; h += nwarps) {
        const int64_t i0 = heads[h], i1 = (h + 1 < n_heads) ? heads[h + 1] : n_exc;
        const int64_t s = (int64_t)(keys[i0] >> 32);
        const uint4* p0 = a.b0 + s * a.Wq;
        const uint4* p1 = a.b1 + s * a.Wq;
        const uint4* pv = a.v + s * a.Wq;
        for (int q = 0; q < a.k; ++q) {
            uint32_t c[PFA_NCLASS];
            pfa_class_counts<true>(p0, p1, pv, a.masks + (int64_t)q * a.Wq, a.Wq, lane, c);
            if (c[PFA_C_ESC] == 0) continue;  // warp-uniform: the main kernel already counted this (site, pop)
            for (int b = lane; b < 256; b += 32) hist[wib][b] = 0u;
            __syncwarp();
            const uint32_t* mq = reinterpret_cast<const uint32_t*>(a.masks + (int64_t)q * a.Wq);
            for (int64_t i = i0 + lane; i < i1; i += 32) {
                const unsigned long long key = keys[i];
                const uint32_t row = (uint32_t)(key & 0xffffffull);
                if ((mq[row >> 5] >> (row & 31)) & 1u) atomicAdd(&hist[wib][(key >> 24) & 0xffu], 1u);
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
            PfaSiteResult r = pfa_site_result(c, a.pop_n[q], distinct, sq);
            if (a.isvar) a.isvar[(int64_t)q * a.ns + s] = (uint8_t)r.isvar;
            if (r.isvar) {
                if (a.hsite) a.hsite[(int64_t)q * a.ns + s] = (int64_t)r.h;
                atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q]), 1ull);
                atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 1), r.h);
                if (r.sfs_bin >= 0)
                    atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + r.sfs_bin), 1ull);
            }
        }
    }
}

// second pass of ONE variable site by the whole warp (see pfa_sites.cuh): w0 / w1 / wv are the site's records in the warp's
// shared-memory slot.  S and H of population q < LPS accumulate in the registers of lane q (the lane with sub == q of the
// first group: pfa_site_gap_finish uses the same registers for the lanes with sub == q of every group).
template <int LPS, bool HAS_V, bool MULTI>
__device__ __forceinline__ void pfa_site_coop(const PfaSiteArgs& a, int64_t s, const uint32_t* w0, const uint32_t* w1, const uint32_t* wv,
                                              int Wn, int lane, unsigned long long* sm_SH, unsigned int* sm_sfs, uint32_t& S_mine,
                                              unsigned long long& H_mine, uint32_t fw, unsigned gcr) {
    const int k = MULTI ? a.k : 1;
    for (int q = 0; q < k; ++q) {
        const uint32_t* mq = reinterpret_cast<const uint32_t*>(MULTI ? a.masks + (int64_t)q * a.Wq : a.umask);
        uint32_t c[PFA_NCLASS];
        pfa_coop_counts<HAS_V>(w0, w1, wv, mq, Wn, lane, c, fw, gcr);
        const PfaSiteResult r = pfa_site_result(c, a.pop_n[q], 0u, 0ull);
        if (r.has_escape) continue;  // finished by pfa_escape_sites_kernel
        if (a.isvar && lane == 0) a.isvar[(int64_t)q * a.ns + s] = (uint8_t)r.isvar;
        if (!r.isvar) continue;
        if (a.hsite && lane == 0) a.hsite[(int64_t)q * a.ns + s] = (int64_t)r.h;
        if (q < LPS) {
            if (lane == q) {
                S_mine += 1u;
                H_mine += r.h;
            }
        } else if (lane == 0) {
            atomicAdd(&sm_SH[2 * q], 1ull);
            atomicAdd(&sm_SH[2 * q + 1], r.h);
        }
        if (r.sfs_bin >= 0 && lane == 0) {
            if (a.sfs_in_smem) atomicAdd(&sm_sfs[a.sfs_off[q] + r.sfs_bin], 1u);
            else atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + r.sfs_bin), 1ull);
        }
    }
}

// A site whose VALID rows all show one base but which has rows that are not valid -- gaps, N, ? -- is a segregating site of the
// reference (a gap is an allele, PolyFastA.py:256-258), and in an alignment with sparse gaps and many rows MOST sites are of this
// kind (10,000 rows, one gap per 10^4 bases: 63 % of the sites).  Its statistics need only the numbers of gap / N / ? rows
// per population, and those rows sit in the chunks of flagged cells, which the group already holds in registers: the
// group finishes the site itself -- two packed popcount sums (pfa_site_gap_counts), one shuffle reduction and the arithmetic
// (pfa_site_gap_apply) -- instead of queueing it for the whole warp.  H = n^2 - (valid^2 + gap^2 + N^2 + ?^2); no SFS bin
// (fewer than two of A, C, G, T: getsfs skips the column).  Populations that hold an escape row here are left to
// pfa_escape_sites_kernel, like everywhere else.
template <int LPS, int ITER, bool MULTI>
__device__ __forceinline__ void pfa_site_gap_counts(const PfaSiteArgs& a, int q, const uint4 (&x0)[ITER], const uint4 (&x1)[ITER],
                                                    const uint4 (&mv)[ITER], const uint4 (&um)[ITER], const int (&cell)[ITER], uint32_t fw,
                                                    int sub, uint32_t& pa, uint32_t& pb) {
    pa = pb = 0u;  // (gap | N << 16), (? | escape << 16) among this lane's rows: a count is at most n <= 20,480
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        if (!((fw >> cell[i]) & 1u)) continue;  // rows that are not valid exist in flagged cells only
        uint4 m4 = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        if (MULTI) {
            const int j = sub + LPS * i;
            m4 = j < a.Wq ? __ldg(a.masks + (int64_t)q * a.Wq + j) : make_uint4(0, 0, 0, 0);
        }
        const uint32_t m[4] = {m4.x, m4.y, m4.z, m4.w}, w0[4] = {x0[i].x, x0[i].y, x0[i].z, x0[i].w},
                       w1[4] = {x1[i].x, x1[i].y, x1[i].z, x1[i].w},
                       iv[4] = {um[i].x ^ mv[i].x, um[i].y ^ mv[i].y, um[i].z ^ mv[i].z, um[i].w ^ mv[i].w};  // rows that are not valid
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t im = MULTI ? (iv[w] & m[w]) : iv[w];
            if (im) {
                pa += (uint32_t)__popc(im & ~w1[w] & ~w0[w]) | ((uint32_t)__popc(im & ~w1[w] & w0[w]) << 16);
                pb += (uint32_t)__popc(im & w1[w] & ~w0[w]) | ((uint32_t)__popc(im & w1[w] & w0[w]) << 16);
            }
        }
    }
}

// STORE_H: store the site's H into a.hsite (the single-population call; with several populations a gap site goes to the
// whole-warp pass when the per-site H is wanted: the store inside the population loop cost the validity-aware multi-population
// kernels 8-18 bytes of spills)
template <int LPS, bool STORE_H>
__device__ __forceinline__ void pfa_site_gap_apply(const PfaSiteArgs& a, int64_t s, int q, uint32_t pa, uint32_t pb, int sub, unsigned gmask,
                                                   unsigned long long* sm_SH, uint32_t& S_mine, unsigned long long& H_mine) {
    pa = pfa_group_add<LPS>(pa, gmask);
    pb = pfa_group_add<LPS>(pb, gmask);
    if (pb >> 16) return;  // escape rows: pfa_escape_sites_kernel counts this (site, population)
    const uint32_t cg = pa & 0xffffu, cn = pa >> 16, cq = pb & 0xffffu;
    const uint32_t nq = (uint32_t)a.pop_n[q], valid = nq - (cg + cn + cq);
    const bool isvar = ((valid ? 1 : 0) + (cg ? 1 : 0) + (cn ? 1 : 0) + (cq ? 1 : 0)) > 1;
    if (a.isvar && sub == 0) a.isvar[(int64_t)q * a.ns + s] = (uint8_t)isvar;
    if (!isvar) return;
    const unsigned long long h = (unsigned long long)nq * nq - ((unsigned long long)valid * valid + (unsigned long long)cg * cg +
                                                                 (unsigned long long)cn * cn + (unsigned long long)cq * cq);
    if (STORE_H && a.hsite && sub == 0) a.hsite[(int64_t)q * a.ns + s] = (int64_t)h;
    if (q < LPS) {
        if (sub == q) {
            S_mine += 1u;
            H_mine += h;
        }
    } else if (sub == 0) {
        atomicAdd(&sm_SH[2 * q], 1ull);
        atomicAdd(&sm_SH[2 * q + 1], h);
    }
}

// TMA variant of the register-resident kernel: the bytes in flight are bounded by shared memory instead of registers.
// Every WARP owns one private shared-memory slot; it holds the records of the consecutive sites of m of the warp's passes
// (contiguous in each plane), fetched with one cp.async.bulk per plane that completes on the slot's mbarrier.
// No block-wide synchronisation: a warp waits for its own slot and runs pass 1 of every site on registers (a group of LPS
// lanes per site).  Variable sites (LPS >= 4): the whole warp takes them one at a time, reading the record back from the slot
// (pfa_site_coop); narrow records handled by 1-2 lanes keep the per-group second pass (every lane has its own site there).
// The slot is refilled once its last pass no longer needs it: right after pass 1 when that pass found no variable site,
// else after their second pass -- every shared-memory read of the slot has then been consumed (its value was used), and a
// proxy fence orders those generic-proxy reads before the bulk copy's async-proxy writes.
template <int LPS, int ITER, bool HAS_V, bool MULTI>
__global__ void __launch_bounds__(512, 1) pfa_site_scan_tma_kernel(const PfaSiteArgs a, int m) {
    constexpr int NT = 512;
    // whole-warp second pass for groups of 4-8 lanes; (half-)warp groups keep it on their registers -- unless the validity plane
    // is read too: three planes held through pass 2 do not fit 128 registers (ptxas: 150-360 bytes of spills), the slot does
    constexpr bool COOP = LPS >= 4 && (LPS <= 8 || HAS_V);
    extern __shared__ __align__(128) unsigned char dyn[];
    constexpr int GW = 32 / LPS;        // sites per warp pass
    constexpr int NPL = HAS_V ? 3 : 2;  // planes read
    constexpr int NWARP = NT / 32;
    const int Wq = a.Wq;
    const unsigned rec = (unsigned)Wq * 16u;  // bytes of one site record in one plane
    const int SPS = GW * m;                   // sites per slot: m passes of the warp (narrow records: keeps a copy >= ~2 KB)
    const unsigned VS = HAS_V ? (a.vs > 0 ? (unsigned)a.vs : (unsigned)SPS) : 0u;  // validity records per slot (pfa_slot_issue)
    const unsigned slot_bytes = (unsigned)pfa_slot_bytes(HAS_V, (unsigned)SPS, VS, rec);
    const bool sparse = HAS_V && a.vflag != nullptr;  // fetch only the flagged cells of the v plane
    const int gc = a.gc;
    const unsigned gcr = pfa_cell_rcp(a.gc * 4);
    unsigned char* ring_base = dyn;
    uint64_t* bars = reinterpret_cast<uint64_t*>(dyn + (size_t)NWARP * slot_bytes);  // [warp]
    unsigned long long* sm_SH = reinterpret_cast<unsigned long long*>(bars + NWARP);
    unsigned int* sm_sfs = reinterpret_cast<unsigned int*>(sm_SH + 2 * a.k);
    if (a.x.world && blockIdx.x == 0 && threadIdx.x == 0) a.x.stamps[5] = pfa_globaltimer();
    for (int i = threadIdx.x; i < 2 * a.k; i += blockDim.x) sm_SH[i] = 0ull;
    if (a.sfs_in_smem)
        for (int i = threadIdx.x; i < a.sfs_bins; i += blockDim.x) sm_sfs[i] = 0u;
    if (threadIdx.x == 0) {
        for (int i = 0; i < NWARP; ++i) pfa_mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sub = lane & (LPS - 1), grp = lane / LPS;
    const unsigned gmask = LPS == 32 ? 0xffffffffu : (((1u << LPS) - 1u) << (lane - sub));
    unsigned char* ring = ring_base + (size_t)wib * slot_bytes;
    uint64_t* bar = bars + wib;
    const int64_t nw = (int64_t)gridDim.x * NWARP;
    const int64_t nblk = (a.ns + SPS - 1) / SPS;                     // blocks of SPS consecutive sites
    const unsigned char* planes[3] = {reinterpret_cast<const unsigned char*>(a.b0), reinterpret_cast<const unsigned char*>(a.b1),
                                      reinterpret_cast<const unsigned char*>(a.v)};
    uint32_t S_mine = 0;               // COOP: S and H of population `sub`
    unsigned long long H_mine = 0ull;

    uint4 um[ITER];
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        const int j = sub + LPS * i;
        um[i] = j < Wq ? __ldg(a.umask + j) : make_uint4(0, 0, 0, 0);
    }
    int cell[ITER];  // the flag bit of each of this lane's chunks
#pragma unroll
    for (int i = 0; i < ITER; ++i) cell[i] = (sub + LPS * i) / gc;
    // The first 7/8 of the blocks are split statically (block gw + i nw is warp gw's i-th), the rest is claimed in chunks from
    // a device-wide counter (PfaClaimer): warps that met few variable sites take more of it.
    // `pend` is the block the NEXT refill will fetch, known one refill ahead so that its validity flags are in registers by then.
    PfaClaimer claim;
    const unsigned gw = blockIdx.x * NWARP + wib, nwu = gridDim.x * NWARP;
    const unsigned rounds = (unsigned)(nblk / nwu) * 7u / 8u;  // static rounds of nwu blocks
    unsigned round = 0;
    if (lane == 0) claim.init(a.work, (unsigned)nblk - rounds * nwu, nwu);
    auto next_block = [&]() -> int {  // all lanes
        if (round < rounds) return (int)(gw + (round++) * nwu);
        const int b = __shfl_sync(0xffffffffu, lane == 0 ? claim.next() : 0, 0);
        return b < 0 ? -1 : b + (int)(rounds * nwu);
    };
    int pend = next_block();
    uint32_t pfl[PFA_VF_REGS];
    auto load_flags = [&]() {
#pragma unroll
        for (int u = 0; u < PFA_VF_REGS; ++u) {
            const int64_t s = (int64_t)pend * SPS + u * 32 + lane;
            pfl[u] = (sparse && pend >= 0 && u * 32 + lane < SPS && s < a.ns) ? __ldg(a.vflag + s) : 0u;
        }
    };
    load_flags();
    bool pend_v = HAS_V, cur_v = HAS_V;  // does the block in the slot (being fetched / being scanned) carry validity pieces?
    auto issue_next = [&]() -> int {  // all lanes: fetch `pend` into the warp's slot, then look one block further ahead
        const int blk = pend;
        if (blk >= 0) {
            const int64_t s0 = (int64_t)blk * SPS;
            pend_v = pfa_slot_issue<HAS_V>(ring, bar, planes[0], planes[1], planes[2], sparse, gc, s0, (unsigned)min((int64_t)SPS, a.ns - s0),
                                           (unsigned)SPS, VS, rec, Wq, pfl, lane);
        }
        pend = blk >= 0 ? next_block() : -1;
        load_flags();
        return blk;
    };
    int cur_blk = issue_next();
    cur_v = pend_v;

    for (unsigned k = 0; cur_blk >= 0; ++k) {
        const int64_t blk = cur_blk;
        const bool bv = cur_v;  // false: no row of this block's sites is invalid -- the two-plane code path
        pfa_mbar_wait(bar, k & 1u);
        const unsigned char* slot = ring;
        auto refill = [&]() {  // once per block, when the slot's last pass no longer needs it
            cur_blk = issue_next();
            cur_v = pend_v;
        };
        for (int t = 0; t < m; ++t) {
            if (COOP) {
                // One pass over GW sites of the slot with the whole-warp second pass.  Blocks without a flagged cell run the
                // two-plane pass 1 even in an alignment that has invalid rows somewhere.  What follows pass 1 is ONE piece of code
                // for both: the kernel's hot loop has to fit the instruction cache (a version with the refill and the second pass
                // inlined per path -- 7,000 instructions -- stalled 6 cycles per issue on instruction fetch, ncu r2w_k2g).
                const int idx = t * GW + grp;  // site of this group inside the slot
                const int64_t s = blk * SPS + idx;
                const uint4* q0 = reinterpret_cast<const uint4*>(slot + (size_t)idx * rec);
                const uint4* q1 = reinterpret_cast<const uint4*>(slot + (size_t)(SPS + idx) * rec);
                const uint32_t* fa = pfa_slot_flags(slot, (unsigned)SPS, VS, rec);  // flag words of the slot's sites (sparse)
                uint4 x0[ITER], x1[ITER];
                // unconditional loads: chunks beyond the record and sites beyond the end read whatever lies there in the slot (the
                // allocation is padded); every use is masked (those chunks' masks are zero) or dropped (s >= ns)
#pragma unroll
                for (int i = 0; i < ITER; ++i) {
                    x0[i] = q0[sub + LPS * i];
                    x1[i] = q1[sub + LPS * i];
                }
                bool var, gapsite = false;
                uint32_t pa = 0, pb = 0;
                if (!(HAS_V && bv)) {
                    const unsigned f = pfa_site_pass1<LPS, ITER, false, false>(x0, x1, um, um, gmask);
                    var = s < a.ns && !pfa_flags_bases_mono(f);
                } else {
                    // a site beyond the end of the shard (last block) has no flag word in the slot: what lies there is stale
                    const uint32_t fw = s >= a.ns ? 0u : sparse ? fa[idx] : 0xffffffffu;
                    const uint4* qv = reinterpret_cast<const uint4*>(
                        pfa_slot_vrec(slot, (unsigned)SPS, VS, rec, sparse, idx, planes[2] + (size_t)(s < a.ns ? s : 0) * rec));
                    uint4 mv[ITER];  // rows of the union that are valid
#pragma unroll
                    for (int i = 0; i < ITER; ++i) {
                        mv[i] = um[i];
                        if ((fw >> cell[i]) & 1u) {
                            const uint4 v4 = qv[sub + LPS * i];
                            mv[i] = make_uint4(um[i].x & v4.x, um[i].y & v4.y, um[i].z & v4.z, um[i].w & v4.w);
                        }
                    }
                    // base-plane flags over the VALID rows: bases_mono = every valid row shows the same base
                    const unsigned f = pfa_site_pass1_valid<LPS, ITER>(x0, x1, mv, um, gmask);
                    const bool bmono = pfa_flags_bases_mono(f);
                    var = s < a.ns && !bmono;
                    gapsite = s < a.ns && bmono && (f & 32u);  // its valid rows show one base, but not all rows are valid
                    if (MULTI && gapsite && a.hsite) {  // per-site H wanted: the whole-warp pass counts and stores it (see pfa_site_gap_apply)
                        var = true;
                        gapsite = false;
                    }
                    if (gapsite) {
                        if (!MULTI) {
                            pfa_site_gap_counts<LPS, ITER, false>(a, 0, x0, x1, mv, um, cell, fw, sub, pa, pb);
                        } else {
                            for (int q = 0; q < a.k; ++q) {
                                pfa_site_gap_counts<LPS, ITER, true>(a, q, x0, x1, mv, um, cell, fw, sub, pa, pb);
                                pfa_site_gap_apply<LPS, false>(a, s, q, pa, pb, sub, gmask, sm_SH, S_mine, H_mine);
                            }
                        }
                    }
                }
                if (a.isvar && sub == 0 && s < a.ns && !var && !gapsite)
                    for (int q = 0; q < a.k; ++q) a.isvar[(int64_t)q * a.ns + s] = 0;
                // variable sites: the whole warp, one at a time, from the slot
                for (unsigned rest = __ballot_sync(0xffffffffu, var && sub == 0); rest; rest &= rest - 1) {
                    const int vidx = t * GW + (__ffs(rest) - 1) / LPS;
                    const uint32_t* r0 = reinterpret_cast<const uint32_t*>(slot + (size_t)vidx * rec);
                    const uint32_t* r1 = reinterpret_cast<const uint32_t*>(slot + (size_t)(SPS + vidx) * rec);
                    const uint32_t fwv = !(HAS_V && bv) ? 0u : sparse ? fa[vidx] : 0xffffffffu;
                    if (HAS_V && fwv)
                        pfa_site_coop<LPS, HAS_V, MULTI>(a, blk * SPS + vidx, r0, r1,
                                                         reinterpret_cast<const uint32_t*>(pfa_slot_vrec(slot, (unsigned)SPS, VS, rec, sparse, vidx, planes[2] + (size_t)(blk * SPS + vidx) * rec)),
                                                         Wq * 4, lane, sm_SH, sm_sfs, S_mine, H_mine, fwv, gcr);
                    else
                        pfa_site_coop<LPS, false, MULTI>(a, blk * SPS + vidx, r0, r1, r0, Wq * 4, lane, sm_SH, sm_sfs, S_mine, H_mine, 0u, 0u);
                }
                // the slot's last pass no longer needs it: fetch the next block; what is left of a gap site runs on registers
                // while that block is on its way
                if (t == m - 1) refill();
                if (HAS_V && !MULTI && gapsite) pfa_site_gap_apply<LPS, true>(a, s, 0, pa, pb, sub, gmask, sm_SH, S_mine, H_mine);
            } else {
                const int idx = t * GW + grp;  // site of this group inside the slot
                const int64_t s = blk * SPS + idx;
                const uint4* q0 = reinterpret_cast<const uint4*>(slot + (size_t)idx * rec);
                const uint4* q1 = reinterpret_cast<const uint4*>(slot + (size_t)(SPS + idx) * rec);
                const uint4* qv = reinterpret_cast<const uint4*>(slot + (size_t)(2 * SPS + idx) * rec);
                uint4 x0[ITER], x1[ITER], xv[ITER];
#pragma unroll
                for (int i = 0; i < ITER; ++i) {
                    const int j = sub + LPS * i;  // unconditional loads, see pfa_site_tma_pass
                    x0[i] = q0[j];
                    x1[i] = q1[j];
                    xv[i] = HAS_V ? qv[j] : um[i];
                }
                // pass 1 has consumed every register loaded from the slot: the slot can be refilled while the second pass (on
                // registers) runs
                const unsigned f = pfa_site_pass1<LPS, ITER, HAS_V>(x0, x1, xv, um, gmask);
                if (t == m - 1) refill();
                if (s < a.ns) pfa_site_finish_regs<LPS, ITER, HAS_V, MULTI>(a, s, f, x0, x1, xv, um, sub, gmask, Wq, sm_SH, sm_sfs);
            }
        }
    }
    if (COOP && sub < a.k && S_mine) {  // population `sub`: whole-warp second passes (first group) and gap sites (every group)
        atomicAdd(&sm_SH[2 * sub], (unsigned long long)S_mine);
        atomicAdd(&sm_SH[2 * sub + 1], H_mine);
    }
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(a.work + 1, 1u) == gridDim.x - 1) {  // every CTA has made its last claim: reset for the next launch
        a.work[0] = 0u;
        a.work[1] = 0u;
    }
    for (int q = threadIdx.x; q < a.k; q += blockDim.x) {
        if (sm_SH[2 * q]) {
            atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q]), sm_SH[2 * q]);
            atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 1), sm_SH[2 * q + 1]);
        }
    }
    if (a.sfs_in_smem) {
        for (int q = 0; q < a.k; ++q) {
            const int nb = (int)(a.pop_n[q] / 2);
            for (int i = threadIdx.x; i < nb; i += blockDim.x) {
                const unsigned int cnt = sm_sfs[a.sfs_off[q] + i];
                if (cnt) atomicAdd(reinterpret_cast<unsigned long long*>(a.out + a.out_off[q] + 2 + i), (unsigned long long)cnt);
            }
        }
    }
    if (a.x.world) pfa_xchg_epilogue(a.x);
}

int pfa_tma_plan(pfa_aln* a, const PfaTmaShape& s, PfaTmaPlan* p) {
    pfa_ctx* ctx = a->ctx;
    const char* m_env = getenv(s.m_env);
    const char* vflag = getenv("PFA_VFLAG");
    const char* vcompact = getenv("PFA_VCOMPACT");
    const char* vdiv = getenv("PFA_VDIV");
    const int gw = 32 / s.lps, nwarp = s.nt / 32;
    const int m_sparse = std::max(1, 32 * PFA_VF_REGS / (s.recs * gw));  // sparse validity: a slot's flag words fit PFA_VF_REGS per lane
    int m = m_env ? std::max(1, atoi(m_env)) : s.m;
    // validity flags: a shard with a few non-ACGT symbols fetches only the flagged pieces of its v plane (pfa_slot_issue); not
    // when the validity plane is forced (benchmarks of the 3-plane worst case) or PFA_VFLAG=0
    p->sparse_v = s.has_v && !(a->has_invalid & 2) && s.lps >= 4 && a->Wq >= 4 && !(vflag && atoi(vflag) == 0);
    if (p->sparse_v) m = std::min(m, m_sparse);
    // sparse validity: the fewer sites are flagged, the smaller the slots' v area and the more shared memory goes into passes per
    // slot -- with two passes per slot the validity-aware K2 runs a clean or nearly clean 10,000-row shard as fast as the
    // pure-ACGT kernel (0.73 against 0.77 ms with one; scripts/probe_gaps5.py), K4 at 2,000 rows two passes instead of one
    p->flagged_sites = 0;
    if (p->sparse_v)
        if (int rc = pfa_aln_flagged_sites(a, &p->flagged_sites)) return rc;
    p->v_div = 1;
    if (p->sparse_v && !(vcompact && atoi(vcompact) == 0))
        for (int d = s.v_div_max; d > 1 && p->v_div == 1; d /= 2)
            if (p->flagged_sites * d * d <= a->ns) p->v_div = d;
    if (p->sparse_v && vdiv) p->v_div = std::max(1, std::min(8, atoi(vdiv)));  // tests: force a small v area
    if (p->v_div > 1 && !m_env) m = std::min(m + (m * s.m_raise + 1) / 2, m_sparse);
    auto vs_for = [&](int mm) { return s.has_v ? std::max(s.recs, s.recs * gw * mm / p->v_div) : 0; };
    auto dyn_for = [&](int mm) {
        return (size_t)nwarp * pfa_slot_bytes(s.has_v, (unsigned)(s.recs * gw * mm), (unsigned)vs_for(mm), (unsigned)a->Wq * 16u) +
               sizeof(uint64_t) * nwarp + s.smem + 1024;  // + slack: unconditional chunk loads may run past the last record
    };
    while (m > 1 && dyn_for(m) > PFA_TMA_SMEM_MAX) --m;
    // At the widest record of either scan (160 chunks) one pass per slot fits for any k below ~6,600 populations.  Above
    // k = 3,072 the register kernels' 16 k bytes of dynamic shared memory passed 48 KB: they could not take this case either.
    if (dyn_for(m) > PFA_TMA_SMEM_MAX)
        return pfa_fail(ctx, PFA_ERR_ARG, "TMA scan: one pass per slot needs %zu bytes of shared memory (k = %d populations, %d chunks per record)",
                        dyn_for(m), a->k, a->Wq);
    p->m = m;
    p->vs = vs_for(m);
    p->dyn = dyn_for(m);
    const int64_t per_cta = (int64_t)gw * m * nwarp;
    p->grid = (unsigned)std::min<int64_t>(ctx->sm_count, (std::max<int64_t>(s.units, 1) + per_cta - 1) / per_cta);
    return PFA_OK;
}

int pfa_launch_site_scan(pfa_aln* a, int64_t* d_out, uint8_t* d_isvar, pfa_xchg* x, bool defer, int64_t* d_hsite) {
    pfa_ctx* ctx = a->ctx;
    const int64_t out_len = a->site_off[a->k];
    if (!x) PFA_CUDA(ctx, cudaMemsetAsync(d_out, 0, sizeof(int64_t) * (size_t)out_len, ctx->stream));
    // per-site H: the kernels store only variable (site, population) pairs, everything else stays zero
    if (d_hsite && a->ns > 0) PFA_CUDA(ctx, cudaMemsetAsync(d_hsite, 0, sizeof(int64_t) * (size_t)a->k * (size_t)a->ns, ctx->stream));
    if (x && defer) {
        if (pfa_xchg_carry(x) != 0 || out_len > pfa_xchg_cap(x)) return pfa_fail(ctx, PFA_ERR_ARG, "deferred exchange: buffer in use or too small");
        pfa_xchg_set_carry(x, out_len);  // the next exchange pushes these words along
        if (a->ns == 0 || a->n == 0) return PFA_OK;
    }
    if (a->ns == 0 || a->n == 0) return x ? pfa_xchg_launch_only(x, nullptr, out_len, d_out) : PFA_OK;
    PfaSiteArgs args;
    unsigned int* work = nullptr;
    if (int rc = pfa_ctx_work(ctx, &work)) return rc;
    pfa_fill_site_args(a, d_out, d_isvar, &args, d_hsite);
    if (x) {
        // the blocks add into the exchange's partial vector (zero between launches); the escape kernel goes FIRST so that
        // the scan kernel's last block sees the complete shard vector when it runs the exchange
        args.out = reinterpret_cast<int64_t*>(pfa_xchg_partial(x));
        if (a->n_exc_sites > 0) {
            int rc = pfa_launch_escape(a, pfa_escape_sites_kernel, args);
            if (rc) return rc;
        }
        if (!defer) {
            int rc = pfa_xchg_fill(x, out_len, d_out, &args.x, true);  // the TMA kernels run one CTA per SM: all blocks may take part
            if (rc) return rc;
        }
    }
    // lanes per site: the smallest power of two that leaves every lane at most 5 chunks
    // (measured over n = 100 ... 10,000, DESIGN.md section 3: fewer chunks per lane with more lanes per site, at higher
    // occupancy, is never faster -- bytes in flight per lane win)
    int lps = 1;
    while (lps < 32 && (a->Wq + lps - 1) / lps > 5) lps *= 2;
    const int iter = (a->Wq + lps - 1) / lps;
    const size_t smem = sizeof(unsigned long long) * 2 * (size_t)a->k + (args.sfs_in_smem ? sizeof(unsigned int) * (size_t)args.sfs_bins : 0);
    const bool hv = a->has_invalid != 0, multi = a->k > 1;
    const bool generic = iter > 5;  // lps = 32: records of more than 160 chunks (n > 20,480) stream through one warp per site
    const char* planes = pfa_plane_alloc_name(a->plane_alloc);
    cudaStream_t st = ctx->stream;
    // The TMA variant: one CTA of 512 threads per SM, every warp fed by cp.async.bulk through its own shared-memory slot of
    // about 5 KB per plane (several passes of the warp for narrow records).  Measured against the register-resident kernel
    // over n = 100 ... 20,000 (DESIGN.md section 3): 1-2 % faster at n = 10,000, 6-20 % at n = 2,000 ... 6,000 and 16,000,
    // ~10 % for n <= 384; slower only for records of 4 ... 10 chunks handled by 1-2 lanes (n = 385 ... 1,280), which stay on
    // the register kernel.
    if (!generic && (lps >= 4 || a->Wq <= 3)) {
        constexpr int nt = 512;
        const int gw = 32 / lps, nwarp = nt / 32;
        const int64_t pass_bytes = (int64_t)gw * a->Wq * 16;  // one pass of a warp, per plane
        // passes per slot: ~5 KB per plane.  Rounded to the nearest when every warp still gets >= 512 blocks (C4 on one GPU, two
        // passes of 2.5 KB: 3.46 ms against 3.55 with one), else rounded down: on a 1.25 Mb shard of C4 (one of 8 GPUs) the larger
        // blocks cost 4 % (0.476 against 0.458 ms), at 5 Mb they break even
        int m = (int)std::max<int64_t>(1, 5000 / pass_bytes);
        const int64_t m_near = std::max<int64_t>(1, (5000 + pass_bytes / 2) / pass_bytes);
        if (m_near > m && a->ns / ((int64_t)gw * m_near * nwarp * ctx->sm_count) >= 512) m = (int)m_near;
        const PfaTmaShape shape = {1, a->ns, lps, nt, m, "PFA_SITE_TMA_M", 4, 2, smem, hv};
        PfaTmaPlan p;
        if (int rc = pfa_tma_plan(a, shape, &p)) return rc;
        if (p.sparse_v) args.vflag = a->vflag;
        args.vs = p.vs;
        const bool found = pfa_for_shape<1, 1, 1, 2, 1, 3, 4, 3, 4, 4, 4, 5, 8, 3, 8, 4, 8, 5, 16, 3, 16, 4, 16, 5, 32, 3, 32, 4, 32, 5>(
            lps, iter, [&](auto L, auto I) {
                pfa_for_v_multi(hv, multi, [&](auto V, auto M) {
                    auto kernel = pfa_site_scan_tma_kernel<decltype(L)::value, decltype(I)::value, decltype(V)::value, decltype(M)::value>;
                    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.dyn);
                    kernel<<<p.grid, nt, p.dyn, st>>>(args, p.m);
                });
            });
        if (!found) return pfa_fail(ctx, PFA_ERR_ARG, "site scan: no TMA kernel for lps=%d iter=%d", lps, iter);
        pfa_note_kernel(ctx, "pfa_site_scan_tma_kernel<LPS=%d,ITER=%d,HAS_V=%d,MULTI=%d> grid=%u block=%d passes_per_slot=%d v_records_per_slot=%d planes=%s",
                        lps, iter, (int)hv, (int)multi, p.grid, nt, p.m, args.vs, planes);
        return pfa_scan_done(a, x, !defer, pfa_escape_sites_kernel, args);
    }
    args.x.wide = 0;  // several CTAs per SM, grids beyond the resident set: the last block alone runs the exchange
    const int64_t groups_per_block = PFA_SITE_THREADS / lps;
    const int64_t blocks = std::min<int64_t>((a->ns + groups_per_block - 1) / groups_per_block, (int64_t)ctx->sm_count * (generic ? 4 : 2));
    const dim3 grid((unsigned)blocks);
    if (generic) {
        if (hv) pfa_site_scan_kernel<true><<<grid, PFA_SITE_THREADS, smem, st>>>(args);
        else pfa_site_scan_kernel<false><<<grid, PFA_SITE_THREADS, smem, st>>>(args);
    } else {
        const bool found = pfa_for_shape<1, 4, 1, 5, 2, 3, 2, 4, 2, 5>(lps, iter, [&](auto L, auto I) {
            pfa_for_v_multi(hv, multi, [&](auto V, auto M) {
                pfa_site_scan_reg_kernel<decltype(L)::value, decltype(I)::value, decltype(V)::value, decltype(M)::value>
                    <<<grid, PFA_SITE_THREADS, smem, st>>>(args);
            });
        });
        if (!found) return pfa_fail(ctx, PFA_ERR_ARG, "site scan: no kernel for lps=%d iter=%d", lps, iter);
    }
    pfa_note_kernel(ctx, "%s<LPS=%d,ITER=%d,HAS_V=%d,MULTI=%d> grid=%u block=%d planes=%s", generic ? "pfa_site_scan_kernel" : "pfa_site_scan_reg_kernel", lps, iter,
                    (int)hv, (int)multi, grid.x, PFA_SITE_THREADS, planes);
    return pfa_scan_done(a, x, !defer, pfa_escape_sites_kernel, args);
}

// ---- measurement aid: how fast can this GPU READ the planes at all? -------------------------------------------------------
// The same streaming 128-bit loads as K2 over the same bytes, nothing else (XOR into a register, one store per thread that
// never happens in practice), 8 loads in flight per thread.  bench.py reports K2 against this read-only ceiling next to the
// read+write copy peak.
__global__ void __launch_bounds__(256) pfa_read_probe_kernel(const uint4* __restrict__ p, int64_t n16, unsigned int* __restrict__ sink) {
    constexpr int UNROLL = 8;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (; i + (UNROLL - 1) * stride < n16; i += UNROLL * stride) {
        uint4 x[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) x[u] = pfa_ld_stream(p + i + u * stride);
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            acc.x ^= x[u].x; acc.y ^= x[u].y; acc.z ^= x[u].z; acc.w ^= x[u].w;
        }
    }
    for (; i < n16; i += stride) {
        const uint4 x = pfa_ld_stream(p + i);
        acc.x ^= x.x; acc.y ^= x.y; acc.z ^= x.z; acc.w ^= x.w;
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x9e3779b9u && acc.x == 0x7f4a7c15u) *sink = acc.x;
}

extern "C" int pfa_aln_read_probe(pfa_aln* a, int planes, int reps, double* ms_per_pass) {
    if (!a || !ms_per_pass || planes < 1 || planes > 3 || reps < 1) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    unsigned int* sink = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &sink, sizeof(unsigned int)));
    cudaEvent_t e0, e1;
    PFA_CUDA(ctx, cudaEventCreate(&e0));
    PFA_CUDA(ctx, cudaEventCreate(&e1));
    const int64_t n16 = (int64_t)(a->plane_bytes / 16) * planes;  // b0 | b1 | v are one allocation
    const unsigned grid = (unsigned)ctx->sm_count * 8u;           // 8 CTAs per SM
    auto launch = [&]() { pfa_read_probe_kernel<<<grid, 256, 0, ctx->stream>>>(a->planes, n16, sink); };
    launch();  // warm-up
    cudaEventRecord(e0, ctx->stream);
    for (int r = 0; r < reps; ++r) launch();
    cudaEventRecord(e1, ctx->stream);
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    pfa_dfree(ctx, sink);
    ctx->launches += reps + 1;
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "read probe: %s", cudaGetErrorString(e));
    *ms_per_pass = ms / reps;
    return PFA_OK;
}
