// K4: codon scan -- synonymous / nonsynonymous site and difference counting as the reference does it.
//
// Replaces getvarCDSsites (PolyFastA.py:284-315), get_syn_nonsyn_cod_sites (:319-434), syncodfreq (:536-557)
// and the var-site matching of print_result (:169-170).  Everything the reference derives from one codon
// column is a function of the SET of clean codons ([ACGT]{3}, stops included) its rows show, i.e. of a 64-bit
// presence mask per population:
//   nstops  += [mask & stops != 0]                                   (:293)
//   missing += 3 when the mask is empty                              (:305; also the trailing partial column)
//   sum3_by_len[popc(mask)] += sum_{c in mask} 3*syncodfreq(c)       (:307, kept as exact integers)
//   labels of the three positions from the sense codons of the mask  (:311, tables in constant memory)
//   S_s/H_s and S_n/H_n: for each labelled position the FULL column's n^2 - sum_a c_a^2 (:169-170)
// A warp owns one codon column (three consecutive site records).  Pass 1 proves, with logic ops
// only, that all three sites are monomorphic over the union of the populations -- then every population sees
// the same single codon and the contribution is uniform.  Otherwise pass 2 builds the presence mask per
// population by peeling distinct codons off each 32-row word, and counts the three columns with popcounts.
#include <algorithm>

#include "pfa_batch.cuh"
#include "pfa_codon_rules.h"
#include "pfa_sites.cuh"

__constant__ uint8_t c_syn3[64];
__constant__ uint8_t c_pair[64 * 64];
__constant__ unsigned long long c_class_mask[24];
__constant__ unsigned long long c_stop_mask;
__constant__ unsigned long long c_syn3_bits[3];  // bit b of 3*syncodfreq(c) at bit c of word b: sums over a codon set are three popcounts
__constant__ int c_num_classes;
__device__ uint8_t g_pair[64 * 64];  // the pair table once more in global memory: lane-divergent lookups (pfa_cds_flush) go through L1

int pfa_upload_codon_tables(pfa_ctx* ctx) {
    const PfaCodonTables& t = pfa_codon_tables();
    unsigned long long cm[24];
    for (int i = 0; i < 24; ++i) cm[i] = t.class_mask[i];
    const unsigned long long sm = t.stop_mask;
    PFA_CUDA(ctx, cudaMemcpyToSymbol(c_syn3, t.syn3, 64));
    PFA_CUDA(ctx, cudaMemcpyToSymbol(c_pair, t.pair, 64 * 64));
    PFA_CUDA(ctx, cudaMemcpyToSymbol(g_pair, t.pair, 64 * 64));
    PFA_CUDA(ctx, cudaMemcpyToSymbol(c_class_mask, cm, sizeof cm));
    PFA_CUDA(ctx, cudaMemcpyToSymbol(c_stop_mask, &sm, sizeof sm));
    unsigned long long sb[3] = {0ull, 0ull, 0ull};
    for (int c = 0; c < 64; ++c)
        for (int b = 0; b < 3; ++b)
            if ((t.syn3[c] >> b) & 1) sb[b] |= 1ull << c;
    PFA_CUDA(ctx, cudaMemcpyToSymbol(c_syn3_bits, sb, sizeof sb));
    PFA_CUDA(ctx, cudaMemcpyToSymbol(c_num_classes, &t.num_classes, sizeof(int)));
    return PFA_OK;
}

struct PfaCdsArgs {
    PfaSiteArgs s;
    int64_t* out;      // [k][PFA_CDS_LEN]
    uint8_t* labels;   // optional [k][ns]
    int64_t ncf;       // complete codon columns in this shard
    int has_partial;   // the shard ends with a partial codon column (1 or 2 sites)
    int acc_in_smem;
    int min_nq;        // rows of the smallest population
};

// what the per-column code needs to know about the alignment (or, on the batched path, about one locus of the batch)
struct PfaCdsView {
    const uint4* masks;     // [k][Wq]
    const int64_t* pop_n;   // [k]
    int64_t* out;           // [k][PFA_CDS_LEN] in global memory
    uint8_t* labels;        // optional [k][ns]
    int64_t ns;
    int k;
    int acc_in_smem;        // accumulate into sm_acc[k][PFA_CDS_LEN] instead of out
};
__device__ __forceinline__ PfaCdsView pfa_cds_view(const PfaCdsArgs& a) {
    return PfaCdsView{a.s.masks, a.s.pop_n, a.out, a.labels, a.s.ns, a.s.k, a.acc_in_smem};
}

// labels of the three codon positions from the set of sense codons of a column (PolyFastA.py:331-432)
template <bool DIVERGENT = false>
__device__ __forceinline__ int pfa_labels_from_set(unsigned long long g) {
    const int n = __popcll(g);
    if (n < 2) return 0;
    if (n == 2) {
        const int i = (__ffsll((long long)g) - 1) * 64 + (63 - __clzll((long long)g));
        return DIVERGENT ? (int)__ldg(&g_pair[i]) : (int)c_pair[i];
    }
    unsigned seen0 = 0, seen1 = 0, seen2 = 0;
    for (unsigned long long t = g; t; t &= t - 1) {
        const int c = __ffsll((long long)t) - 1;
        seen0 |= 1u << (c >> 4);
        seen1 |= 1u << ((c >> 2) & 3);
        seen2 |= 1u << (c & 3);
    }
    const int nb[3] = {__popc(seen0), __popc(seen1), __popc(seen2)};
    int top = 0;
    for (int k = 0; k < c_num_classes; ++k) top = max(top, __popcll(g & c_class_mask[k]));
    int last = nb[2] > 1 ? 2 : nb[1] > 1 ? 1 : 0;
    int lab[3] = {0, 0, 0};
    if (top >= 2) {  // some class repeats (:417-429)
        for (int i = 0; i < last; ++i)
            if (nb[i] > 1) lab[i] = 2;
        if (top >= nb[last]) lab[last] = 1;
    } else {  // :432
        for (int i = 0; i < 3; ++i)
            if (nb[i] > 1) lab[i] = 2;
    }
    return lab[0] | (lab[1] << 2) | (lab[2] << 4);
}

// presence mask of clean codons among the rows of one population, OR-reduced over the warp
template <bool HAS_V>
__device__ __forceinline__ unsigned long long pfa_codon_presence(const uint4* __restrict__ b0, const uint4* __restrict__ b1,
                                                                  const uint4* __restrict__ v, int64_t site, int Wq,
                                                                  const uint4* __restrict__ mq, int lane) {
    unsigned long long P = 0;
    const uint32_t* q0 = reinterpret_cast<const uint32_t*>(b0 + site * Wq);
    const uint32_t* q1 = reinterpret_cast<const uint32_t*>(b1 + site * Wq);
    const uint32_t* qv = reinterpret_cast<const uint32_t*>(v + site * Wq);
    const uint32_t* qm = reinterpret_cast<const uint32_t*>(mq);
    const int Wn = Wq * 4;
    for (int j = lane; j < Wq; j += 32) {
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int o = j * 4 + w;
            uint32_t live = __ldg(qm + o);
            if (!live) continue;
            uint32_t x[6];
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                x[2 * t] = __ldg(q1 + o + t * Wn);      // high bit of the base at codon position t
                x[2 * t + 1] = __ldg(q0 + o + t * Wn);  // low bit
                if (HAS_V) live &= __ldg(qv + o + t * Wn);
            }
            while (live) {  // peel one distinct codon per iteration
                const int r = __ffs(live) - 1;
                uint32_t match = live;
                int c = 0;
#pragma unroll
                for (int t = 0; t < 6; ++t) {
                    const uint32_t bit = (x[t] >> r) & 1u;
                    c = (c << 1) | (int)bit;
                    match &= x[t] ^ (bit - 1u);
                }
                P |= 1ull << c;
                live &= ~match;
            }
        }
    }
    const uint32_t lo = __reduce_or_sync(0xffffffffu, (uint32_t)P), hi = __reduce_or_sync(0xffffffffu, (uint32_t)(P >> 32));
    return ((unsigned long long)hi << 32) | lo;
}

// everything one (codon column, population) contributes, given its presence mask and the class counts of its sites
__device__ __forceinline__ void pfa_cds_contribute(unsigned long long P, const uint32_t cnt[3][PFA_NCLASS], int64_t nq,
                                                   const uint32_t escd[3], const unsigned long long escsq[3],
                                                   unsigned long long* acc, uint8_t* labels, int64_t site0) {
    if (P & c_stop_mask) atomicAdd(&acc[PFA_CDS_NSTOPS], 1ull);
    const int len = __popcll(P);
    if (len == 0) {
        atomicAdd(&acc[PFA_CDS_MISSING], 3ull);
        return;
    }
    unsigned tot3 = 0;
    for (unsigned long long t = P; t; t &= t - 1) tot3 += c_syn3[__ffsll((long long)t) - 1];
    if (tot3) atomicAdd(&acc[PFA_CDS_SUM3 + len], (unsigned long long)tot3);
    if (len < 2) return;
    const int lab = pfa_labels_from_set(P & ~c_stop_mask);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int li = (lab >> (2 * i)) & 3;
        if (!li) continue;
        const PfaSiteResult r = pfa_site_result(cnt[i], nq, escd[i], escsq[i]);
        atomicAdd(&acc[li == 1 ? PFA_CDS_SS : PFA_CDS_SN], 1ull);
        atomicAdd(&acc[li == 1 ? PFA_CDS_HS : PFA_CDS_HN], r.h);
        if (labels) labels[site0 + i] = (uint8_t)li;
    }
}

// the same for a column in which only position tv varies (c = class counts of that site): no other position can be labelled
__device__ __forceinline__ void pfa_cds_contribute_one(unsigned long long P, const uint32_t c[PFA_NCLASS], int tv, int64_t nq,
                                                       unsigned long long* acc, uint8_t* labels, int64_t site0) {
    if (P & c_stop_mask) atomicAdd(&acc[PFA_CDS_NSTOPS], 1ull);
    const int len = __popcll(P);
    if (len == 0) {
        atomicAdd(&acc[PFA_CDS_MISSING], 3ull);
        return;
    }
    unsigned tot3 = 0;
    for (unsigned long long t = P; t; t &= t - 1) tot3 += c_syn3[__ffsll((long long)t) - 1];
    if (tot3) atomicAdd(&acc[PFA_CDS_SUM3 + len], (unsigned long long)tot3);
    if (len < 2) return;
    const int li = (pfa_labels_from_set(P & ~c_stop_mask) >> (2 * tv)) & 3;
    if (!li) return;
    const PfaSiteResult r = pfa_site_result(c, nq, 0u, 0ull);
    atomicAdd(&acc[li == 1 ? PFA_CDS_SS : PFA_CDS_SN], 1ull);
    atomicAdd(&acc[li == 1 ? PFA_CDS_HS : PFA_CDS_HN], r.h);
    if (labels) labels[site0 + tv] = (uint8_t)li;
}

template <bool HAS_V>
__global__ void __launch_bounds__(PFA_SITE_THREADS) pfa_cds_scan_kernel(const PfaCdsArgs a) {
    extern __shared__ unsigned long long smem[];  // [3] uniform + [k][PFA_CDS_LEN] when acc_in_smem
    const int nacc = 3 + (a.acc_in_smem ? a.s.k * PFA_CDS_LEN : 0);
    for (int i = threadIdx.x; i < nacc; i += blockDim.x) smem[i] = 0ull;
    __syncthreads();
    unsigned long long* sm_acc = smem + 3;

    const int lane = threadIdx.x & 31;
    const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const int64_t nwarps = (int64_t)gridDim.x * blockDim.x / 32;
    const int Wq = a.s.Wq;
    unsigned u_nstops = 0, u_missing = 0, u_sum3 = 0;  // contributions identical for every population

    for (int64_t cc = wid; cc < a.ncf; cc += nwarps) {
        const int64_t site0 = cc * 3;
        // ---- pass 1: are the three sites monomorphic over the union of the populations? ----
        uint32_t acc[3][6];
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
            for (int i = 0; i < 6; ++i) acc[t][i] = 0;
        for (int j = lane; j < Wq; j += 32) {
            const uint4 m = __ldg(a.s.umask + j);
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                const uint4 x0 = pfa_ld_stream(a.s.b0 + (site0 + t) * Wq + j);
                const uint4 x1 = pfa_ld_stream(a.s.b1 + (site0 + t) * Wq + j);
                acc[t][0] |= (x0.x & m.x) | (x0.y & m.y) | (x0.z & m.z) | (x0.w & m.w);
                acc[t][1] |= (~x0.x & m.x) | (~x0.y & m.y) | (~x0.z & m.z) | (~x0.w & m.w);
                acc[t][2] |= (x1.x & m.x) | (x1.y & m.y) | (x1.z & m.z) | (x1.w & m.w);
                acc[t][3] |= (~x1.x & m.x) | (~x1.y & m.y) | (~x1.z & m.z) | (~x1.w & m.w);
                if (HAS_V) {
                    const uint4 xv = pfa_ld_stream(a.s.v + (site0 + t) * Wq + j);
                    acc[t][4] |= (xv.x & m.x) | (xv.y & m.y) | (xv.z & m.z) | (xv.w & m.w);
                    acc[t][5] |= (~xv.x & m.x) | (~xv.y & m.y) | (~xv.z & m.z) | (~xv.w & m.w);
                } else {
                    acc[t][4] |= m.x | m.y | m.z | m.w;
                }
            }
        }
        unsigned f = 0;
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
            for (int i = 0; i < 6; ++i) f |= (acc[t][i] ? 1u : 0u) << (6 * t + i);
        f = __reduce_or_sync(0xffffffffu, f);
        bool uniform = true, clean = true;
        int codon = 0;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const unsigned ft = (f >> (6 * t)) & 63u;
            const bool mono = ((ft & 3u) != 3u) && ((ft & 12u) != 12u) && ((ft & 48u) != 48u);
            const bool all_escape = (ft & 1u) && (ft & 4u) && !(ft & 16u);
            uniform = uniform && mono && !all_escape;
            clean = clean && (ft & 16u) && !(ft & 32u);
            codon = (codon << 2) | ((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0);
        }
        if (uniform) {
            if (lane == 0) {
                if (clean) {
                    u_nstops += (unsigned)((c_stop_mask >> codon) & 1ull);
                    u_sum3 += c_syn3[codon];
                } else {
                    u_missing += 3;
                }
            }
            continue;
        }
        // ---- pass 2: per population ----
        for (int q = 0; q < a.s.k; ++q) {
            const uint4* mq = a.s.masks + (int64_t)q * Wq;
            uint32_t cnt[3][PFA_NCLASS];
#pragma unroll
            for (int t = 0; t < 3; ++t)
                pfa_class_counts<HAS_V>(a.s.b0 + (site0 + t) * Wq, a.s.b1 + (site0 + t) * Wq, a.s.v + (site0 + t) * Wq, mq, Wq, lane,
                                        cnt[t]);
            if (cnt[0][PFA_C_ESC] | cnt[1][PFA_C_ESC] | cnt[2][PFA_C_ESC]) continue;  // finished by pfa_cds_escape_kernel
            const unsigned long long P = pfa_codon_presence<HAS_V>(a.s.b0, a.s.b1, a.s.v, site0, Wq, mq, lane);
            if (lane != 0) continue;
            const uint32_t escd[3] = {0, 0, 0};
            const unsigned long long escsq[3] = {0, 0, 0};
            unsigned long long* dst = a.acc_in_smem ? sm_acc + q * PFA_CDS_LEN
                                                    : reinterpret_cast<unsigned long long*>(a.out + (int64_t)q * PFA_CDS_LEN);
            pfa_cds_contribute(P, cnt, a.s.pop_n[q], escd, escsq, dst, a.labels ? a.labels + (int64_t)q * a.s.ns : nullptr, site0);
        }
    }
    if (a.has_partial && blockIdx.x == 0 && threadIdx.x == 0) u_missing += 3;  // :305 for the trailing 1-2 sites
    // ---- flush ----
    for (int off = 16; off; off >>= 1) {
        u_nstops += __shfl_xor_sync(0xffffffffu, u_nstops, off);
        u_missing += __shfl_xor_sync(0xffffffffu, u_missing, off);
        u_sum3 += __shfl_xor_sync(0xffffffffu, u_sum3, off);
    }
    if (lane == 0) {
        if (u_nstops) atomicAdd(&smem[0], (unsigned long long)u_nstops);
        if (u_missing) atomicAdd(&smem[1], (unsigned long long)u_missing);
        if (u_sum3) atomicAdd(&smem[2], (unsigned long long)u_sum3);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < a.s.k * PFA_CDS_LEN; i += blockDim.x) {
        const int e = i % PFA_CDS_LEN;
        unsigned long long x = a.acc_in_smem ? sm_acc[i] : 0ull;
        if (e == PFA_CDS_NSTOPS) x += smem[0];
        if (e == PFA_CDS_MISSING) x += smem[1];
        if (e == PFA_CDS_SUM3 + 1) x += smem[2];
        if (x) atomicAdd(reinterpret_cast<unsigned long long*>(a.out) + i, x);
    }
    if (a.s.x.world) pfa_xchg_epilogue(a.s.x);
}

__device__ __forceinline__ uint32_t pfa_u4(const uint4& x, int w) { return w == 0 ? x.x : w == 1 ? x.y : w == 2 ? x.z : x.w; }

// pass 1 of one codon column whose three site records are in registers: 18 flag bits (6 per site), OR-reduced over the group
// f2 (optional, with HAS_V): 4 more bits per site -- plane b0 / b1 shows a one / a zero among the VALID rows -- which tell a
// column whose only "variation" is missing data (every valid row of a site shows the same base) from real base variation
template <int LPS, int ITER, bool HAS_V>
__device__ __forceinline__ unsigned pfa_cds_pass1(const uint4 (&x0)[3][ITER], const uint4 (&x1)[3][ITER], const uint4 (&xv)[3][ITER],
                                                  const uint4 (&um)[ITER], unsigned gmask) {
    unsigned f = 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        uint32_t o0 = 0, z0 = 0, o1 = 0, z1 = 0, ov = 0, zv = 0;
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            const uint4 m = um[i];
            o0 |= (x0[t][i].x & m.x) | (x0[t][i].y & m.y) | (x0[t][i].z & m.z) | (x0[t][i].w & m.w);
            z0 |= (~x0[t][i].x & m.x) | (~x0[t][i].y & m.y) | (~x0[t][i].z & m.z) | (~x0[t][i].w & m.w);
            o1 |= (x1[t][i].x & m.x) | (x1[t][i].y & m.y) | (x1[t][i].z & m.z) | (x1[t][i].w & m.w);
            z1 |= (~x1[t][i].x & m.x) | (~x1[t][i].y & m.y) | (~x1[t][i].z & m.z) | (~x1[t][i].w & m.w);
            ov |= (xv[t][i].x & m.x) | (xv[t][i].y & m.y) | (xv[t][i].z & m.z) | (xv[t][i].w & m.w);
            if (HAS_V) zv |= (~xv[t][i].x & m.x) | (~xv[t][i].y & m.y) | (~xv[t][i].z & m.z) | (~xv[t][i].w & m.w);
        }
        f |= ((o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (ov ? 16u : 0u) | (zv ? 32u : 0u)) << (6 * t);
    }
    return pfa_group_or<LPS>(f, gmask);
}

// everything after pass 1 of one codon column whose three site records are in registers (f: the 18 flag bits of pass 1);
// shared by the TMA kernel's per-group path and the batched kernel
template <int LPS, int ITER, bool HAS_V, bool MULTI>
__device__ __forceinline__ void pfa_cds_finish_regs(const PfaCdsView& a, int64_t site0, unsigned f, const uint4 (&x0)[3][ITER],
                                                    const uint4 (&x1)[3][ITER], const uint4 (&xv)[3][ITER], const uint4 (&um)[ITER], int sub,
                                                    unsigned gmask, int Wq, unsigned long long* sm_acc, unsigned& u_nstops, unsigned& u_missing,
                                                    unsigned& u_sum3) {
    constexpr bool one_pop = !MULTI;  // one population: its mask is the union mask
    bool uniform = true, clean = true;
    int codon = 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const unsigned ft = (f >> (6 * t)) & 63u;
        const bool mono = ((ft & 3u) != 3u) && ((ft & 12u) != 12u) && ((ft & 48u) != 48u);
        const bool all_escape = (ft & 1u) && (ft & 4u) && !(ft & 16u);
        uniform = uniform && mono && !all_escape;
        clean = clean && (ft & 16u) && !(ft & 32u);
        codon = (codon << 2) | ((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0);
    }
    if (uniform) {
        if (sub == 0) {
            if (clean) {
                u_nstops += (unsigned)((c_stop_mask >> codon) & 1ull);
                u_sum3 += c_syn3[codon];
            } else {
                u_missing += 3;
            }
        }
        return;
    }
    // ---- pass 2, common case: exactly ONE of the three sites varies and the other two show one valid base.  Then the
    // clean codons of a population are that fixed pair combined with the bases present at the variable site, so the
    // presence mask follows from the four base counts of ONE column (no codon peeling, a third of the popcounts); only
    // the variable position can carry a label (a label needs codons that differ there). ----
    int nvar = 0, tv = 0, fixed = 0;
    bool fixed_valid = true;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const unsigned ft = (f >> (6 * t)) & 63u;
        const bool mono = ((ft & 3u) != 3u) && ((ft & 12u) != 12u) && ((ft & 48u) != 48u);
        if (!mono) {
            ++nvar;
            tv = t;
        } else {
            fixed_valid = fixed_valid && (ft & 16u) && !(ft & 32u);
            fixed |= (((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0)) << (2 * (2 - t));
        }
    }
    if (nvar == 1 && fixed_valid) {
        uint32_t mine[PFA_NCLASS];
        int myq = -1;
        auto finish_one = [&](int q, const uint32_t (&c)[PFA_NCLASS]) {
            const int shift = 2 * (2 - tv);
            unsigned long long P = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if (c[b]) P |= 1ull << (fixed | (b << shift));
            unsigned long long* dst = a.acc_in_smem ? sm_acc + q * PFA_CDS_LEN
                                                    : reinterpret_cast<unsigned long long*>(a.out + (int64_t)q * PFA_CDS_LEN);
            pfa_cds_contribute_one(P, c, tv, a.pop_n[q], dst, a.labels ? a.labels + (int64_t)q * a.ns : nullptr, site0);
        };
        for (int q = 0; q < a.k; ++q) {
            const uint4* mq = a.masks + (int64_t)q * Wq;
            uint32_t c[PFA_NCLASS];
#pragma unroll
            for (int i = 0; i < PFA_NCLASS; ++i) c[i] = 0;
#pragma unroll
            for (int i = 0; i < ITER; ++i) {
                const int j = sub + LPS * i;
                uint4 m4 = um[i];
                if (!one_pop) m4 = j < Wq ? __ldg(mq + j) : make_uint4(0, 0, 0, 0);
                const uint4 s0 = tv == 0 ? x0[0][i] : tv == 1 ? x0[1][i] : x0[2][i];
                const uint4 s1 = tv == 0 ? x1[0][i] : tv == 1 ? x1[1][i] : x1[2][i];
                const uint4 sv = tv == 0 ? xv[0][i] : tv == 1 ? xv[1][i] : xv[2][i];
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const uint32_t m = pfa_u4(m4, w), w0 = pfa_u4(s0, w), w1 = pfa_u4(s1, w), wv = pfa_u4(sv, w);
                    const uint32_t vm = HAS_V ? (wv & m) : m;
                    const uint32_t hi = vm & w1, lo = vm & ~w1;
                    c[PFA_C_T] += __popc(hi & w0);
                    c[PFA_C_G] += __popc(hi & ~w0);
                    c[PFA_C_C] += __popc(lo & w0);
                    c[PFA_C_A] += __popc(lo & ~w0);
                    if (HAS_V) {
                        const uint32_t im = ~wv & m;
                        const uint32_t ihi = im & w1;
                        c[PFA_C_ESC] += __popc(ihi & w0);
                        c[PFA_C_Q] += __popc(ihi & ~w0);
                        c[PFA_C_N] += __popc(im & ~w1 & w0);
                    }
                }
            }
            if (LPS > 1) {
#pragma unroll
                for (int i = 0; i < PFA_NCLASS; ++i)
                    if (HAS_V || i < 4) c[i] = pfa_group_add<LPS>(c[i], gmask);
            }
            if (c[PFA_C_ESC]) continue;  // finished by pfa_cds_escape_kernel (group-uniform: every lane holds the sums)
            if (one_pop) {
                if (sub == 0) finish_one(0, c);
                return;
            }
            // several populations: lane q of the group keeps population q's counts, the scalar parts run side by side
            if (sub == (q & (LPS - 1))) {
                if (myq >= 0) finish_one(myq, mine);
#pragma unroll
                for (int i = 0; i < PFA_NCLASS; ++i) mine[i] = c[i];
                myq = q;
            }
        }
        if (myq >= 0) finish_one(myq, mine);
        return;
    }
    // ---- pass 2, general case ----
    for (int q = 0; q < a.k; ++q) {
        const uint4* mq = a.masks + (int64_t)q * Wq;
        uint4 m4[ITER];
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            const int j = sub + LPS * i;
            m4[i] = um[i];
            if (!one_pop) m4[i] = j < Wq ? __ldg(mq + j) : make_uint4(0, 0, 0, 0);
        }
        uint32_t cnt[3][PFA_NCLASS];
        unsigned long long P = 0;
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
            for (int c = 0; c < PFA_NCLASS; ++c) cnt[t][c] = 0;
#pragma unroll
        for (int i = 0; i < ITER; ++i)
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const uint32_t m = pfa_u4(m4[i], w);
                uint32_t live = m;
                uint32_t x[6];
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const uint32_t w0 = pfa_u4(x0[t][i], w), w1 = pfa_u4(x1[t][i], w), wv = pfa_u4(xv[t][i], w);
                    const uint32_t vm = HAS_V ? (wv & m) : m;
                    const uint32_t hi = vm & w1, lo = vm & ~w1;
                    cnt[t][PFA_C_T] += __popc(hi & w0);
                    cnt[t][PFA_C_G] += __popc(hi & ~w0);
                    cnt[t][PFA_C_C] += __popc(lo & w0);
                    cnt[t][PFA_C_A] += __popc(lo & ~w0);
                    if (HAS_V) {
                        const uint32_t im = ~wv & m;
                        const uint32_t ihi = im & w1;
                        cnt[t][PFA_C_ESC] += __popc(ihi & w0);
                        cnt[t][PFA_C_Q] += __popc(ihi & ~w0);
                        cnt[t][PFA_C_N] += __popc(im & ~w1 & w0);
                        live &= wv;
                    }
                    x[2 * t] = w1;
                    x[2 * t + 1] = w0;
                }
                while (live) {  // peel one distinct codon per iteration
                    const int r = __ffs(live) - 1;
                    uint32_t match = live;
                    int c = 0;
#pragma unroll
                    for (int t = 0; t < 6; ++t) {
                        const uint32_t bit = (x[t] >> r) & 1u;
                        c = (c << 1) | (int)bit;
                        match &= x[t] ^ (bit - 1u);
                    }
                    P |= 1ull << c;
                    live &= ~match;
                }
            }
        if (LPS > 1) {
#pragma unroll
            for (int t = 0; t < 3; ++t)
#pragma unroll
                for (int c = 0; c < PFA_NCLASS; ++c)
                    if (HAS_V || c < 4) cnt[t][c] = pfa_group_add<LPS>(cnt[t][c], gmask);
            uint32_t lo = (uint32_t)P, hi = (uint32_t)(P >> 32);
            lo = pfa_group_or<LPS>(lo, gmask);
            hi = pfa_group_or<LPS>(hi, gmask);
            P = ((unsigned long long)hi << 32) | lo;
        }
        if (cnt[0][PFA_C_ESC] | cnt[1][PFA_C_ESC] | cnt[2][PFA_C_ESC]) continue;  // finished by pfa_cds_escape_kernel
        if (sub != 0) continue;
        const uint32_t escd[3] = {0, 0, 0};
        const unsigned long long escsq[3] = {0, 0, 0};
        unsigned long long* dst = a.acc_in_smem ? sm_acc + q * PFA_CDS_LEN
                                                : reinterpret_cast<unsigned long long*>(a.out + (int64_t)q * PFA_CDS_LEN);
        pfa_cds_contribute(P, cnt, a.pop_n[q], escd, escsq, dst, a.labels ? a.labels + (int64_t)q * a.ns : nullptr, site0);
    }
}


template <int LPS, int ITER, bool HAS_V, bool MULTI>
__device__ __forceinline__ void pfa_cds_process(const PfaCdsView& a, int64_t site0, const uint4 (&x0)[3][ITER], const uint4 (&x1)[3][ITER],
                                                const uint4 (&xv)[3][ITER], const uint4 (&um)[ITER], int sub, unsigned gmask, int Wq,
                                                unsigned long long* sm_acc, unsigned& u_nstops, unsigned& u_missing, unsigned& u_sum3) {
    const unsigned f = pfa_cds_pass1<LPS, ITER, HAS_V>(x0, x1, xv, um, gmask);
    pfa_cds_finish_regs<LPS, ITER, HAS_V, MULTI>(a, site0, f, x0, x1, xv, um, sub, gmask, Wq, sm_acc, u_nstops, u_missing, u_sum3);
}

// ---- deferred bookkeeping of the variable codon columns ---------------------------------------------------------------------
// What a (variable codon column, population) contributes is a chain of dependent scalar steps -- stop test, number of clean
// codons, syn-site sum, S/N labels (table lookups), five or six accumulator updates.  Run right after the counts it costs
// the warp ~2,000 cycles per entry with nothing else to overlap (measured: the second population of C3 cost K4 0.06 ms).
// Instead the warp appends (presence mask, H of the three columns, population, site) to a queue of 32 entries in shared
// memory and, when the queue is full (and once at the end), finishes all 32 side by side, one lane each; lanes of the same
// population then combine their terms (match.any + redux) so that one lane per population touches the accumulators.
#define PFA_CDS_QFIELDS 7  // P lo, P hi, h0, h1, h2, population, first site of the column

__device__ __forceinline__ void pfa_cds_enqueue(uint32_t* qbuf, int& count, int lane, unsigned long long P, uint32_t h0, uint32_t h1,
                                                uint32_t h2, int q, uint32_t site0) {
    if (lane < PFA_CDS_QFIELDS) {
        const uint32_t val = lane == 0 ? (uint32_t)P : lane == 1 ? (uint32_t)(P >> 32) : lane == 2 ? h0 : lane == 3 ? h1 : lane == 4 ? h2
                             : lane == 5 ? (uint32_t)q : site0;
        qbuf[lane * 32 + count] = val;
    }
    ++count;
}

// acc: the accumulators [k][PFA_CDS_LEN] (shared or global memory); labels_base: optional [k][ns]
__device__ __noinline__ void pfa_cds_flush(const uint32_t* qbuf, int count, int lane, unsigned long long* acc, uint8_t* labels_base, int64_t ns) {
    __syncwarp();
    const unsigned act = __ballot_sync(0xffffffffu, lane < count);
    if (lane >= count) return;
    const unsigned long long P = ((unsigned long long)qbuf[32 + lane] << 32) | qbuf[lane];
    const uint32_t h[3] = {qbuf[64 + lane], qbuf[96 + lane], qbuf[128 + lane]};
    const int q = (int)qbuf[160 + lane];
    const int64_t site0 = (int64_t)qbuf[192 + lane];
    unsigned long long* dst = acc + (int64_t)q * PFA_CDS_LEN;
    const unsigned stop = (P & c_stop_mask) ? 1u : 0u;
    const int len = __popcll(P);
    unsigned miss = 0, ss = 0, sn = 0, tot3 = 0;
    unsigned long long hs = 0ull, hn = 0ull;
    if (len == 0) {
        miss = 3;
    } else {
        tot3 = (unsigned)__popcll(P & c_syn3_bits[0]) + 2u * (unsigned)__popcll(P & c_syn3_bits[1]) + 4u * (unsigned)__popcll(P & c_syn3_bits[2]);
        if (len >= 2) {
            const int lab = pfa_labels_from_set<true>(P & ~c_stop_mask);
            uint8_t* labels = labels_base ? labels_base + (int64_t)q * ns : nullptr;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int li = (lab >> (2 * i)) & 3;
                if (li == 1) { ss += 1; hs += h[i]; }
                if (li == 2) { sn += 1; hn += h[i]; }
                if (li && labels) labels[site0 + i] = (uint8_t)li;
            }
        }
    }
    // lanes of the same population add up their terms; H in two halves (32 x 3 x n^2 does not fit 32 bits)
    const unsigned peers = __match_any_sync(act, q);
    const unsigned stop_s = __reduce_add_sync(peers, stop), miss_s = __reduce_add_sync(peers, miss);
    const unsigned ss_s = __reduce_add_sync(peers, ss), sn_s = __reduce_add_sync(peers, sn);
    const unsigned long long hs_s = ((unsigned long long)__reduce_add_sync(peers, (unsigned)(hs >> 16)) << 16) + __reduce_add_sync(peers, (unsigned)(hs & 0xffffu));
    const unsigned long long hn_s = ((unsigned long long)__reduce_add_sync(peers, (unsigned)(hn >> 16)) << 16) + __reduce_add_sync(peers, (unsigned)(hn & 0xffffu));
    if (lane == __ffs(peers) - 1) {
        if (stop_s) atomicAdd(&dst[PFA_CDS_NSTOPS], (unsigned long long)stop_s);
        if (miss_s) atomicAdd(&dst[PFA_CDS_MISSING], (unsigned long long)miss_s);
        if (ss_s) { atomicAdd(&dst[PFA_CDS_SS], (unsigned long long)ss_s); atomicAdd(&dst[PFA_CDS_HS], hs_s); }
        if (sn_s) { atomicAdd(&dst[PFA_CDS_SN], (unsigned long long)sn_s); atomicAdd(&dst[PFA_CDS_HN], hn_s); }
    }
    // sum3_by_len: lanes of the same (population, number of clean codons)
    const unsigned peers2 = __match_any_sync(act, (q << 7) | len);
    const unsigned t3 = __reduce_add_sync(peers2, tot3);
    if (t3 && lane == __ffs(peers2) - 1) atomicAdd(&dst[PFA_CDS_SUM3 + len], (unsigned long long)t3);
}

// n^2 - sum_a c_a^2 of one column in 32-bit arithmetic (n < 65536), 0 when the rows show one symbol
__device__ __forceinline__ uint32_t pfa_site_h32(const uint32_t c[PFA_NCLASS], uint32_t nq) {
    uint32_t sum = 0, sq = 0, top = 0;
#pragma unroll
    for (int i = 0; i < PFA_NCLASS; ++i) {
        if (i == PFA_C_ESC) continue;  // columns with escape symbols never come here
        sum += c[i];
        sq += c[i] * c[i];
        top = max(top, c[i]);
    }
    const uint32_t gap = nq - sum;
    sq += gap * gap;
    top = max(top, gap);
    return top == nq ? 0u : nq * nq - sq;
}

// second pass of ONE variable codon column by the whole warp (pfa_sites.cuh): r0 / r1 / rv point to the record of the
// column's first site in the warp's shared-memory slot (32-bit words; the next site follows Wn words later), rv[t] to the
// validity record of site t (pfa_slot_vrec: the three need not be neighbours); f = the 18
// flag bits of pass 1 (6 per site)
template <bool HAS_V, bool MULTI>
__device__ __forceinline__ void pfa_cds_coop(const PfaCdsArgs& a, int64_t site0, unsigned f, const uint32_t* r0, const uint32_t* r1,
                                             const uint32_t* const (&rv)[3], int Wn, int lane, unsigned long long* sm_acc, uint32_t* qbuf, int& qcount,
                                             const uint32_t (&fw)[3], int gcw, unsigned f2) {
    // Missing data only: at each of the three sites the valid rows show ONE base, and the rows that are not valid sit in a few
    // flagged cells.  The rows valid at all three sites then carry one and the same codon: the presence mask has at most that
    // one member (no labels), and only the flagged cells are read -- gaps aligned to codons and runs of N, the usual
    // content of a real CDS alignment, no longer cost the peeling pass over the whole record.
    const uint32_t fwu = fw[0] | fw[1] | fw[2];
    const unsigned gcr = pfa_cell_rcp(gcw);
    bool gaps_only = HAS_V && __popc(fwu) <= 6;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const unsigned g = (f2 >> (4 * t)) & 15u;
        gaps_only = gaps_only && ((g & 3u) != 3u) && ((g & 12u) != 12u);
    }
    if (gaps_only) {
        int codon = 0;
#pragma unroll
        for (int t = 0; t < 3; ++t) codon = (codon << 2) | (((f2 >> (4 * t)) & 4u) ? 2 : 0) | (((f2 >> (4 * t)) & 1u) ? 1 : 0);
        const int kq = MULTI ? a.s.k : 1;
        for (int q = 0; q < kq; ++q) {
            const uint32_t* mq = reinterpret_cast<const uint32_t*>(MULTI ? a.s.masks + (int64_t)q * a.s.Wq : a.s.umask);
            uint32_t ninv = 0, nesc = 0;
            for (uint32_t cells = fwu; cells; cells &= cells - 1) {
                const int cell = __ffs(cells) - 1, w = cell * gcw + lane;
                if (lane < gcw && w < Wn) {
                    const uint32_t m = __ldg(mq + w);
                    uint32_t any = 0;
#pragma unroll
                    for (int t = 0; t < 3; ++t)
                        if ((fw[t] >> cell) & 1u) {
                            const uint32_t inv = ~rv[t][w] & m;
                            any |= inv;
                            nesc += __popc(inv & r1[t * Wn + w] & r0[t * Wn + w]);
                        }
                    ninv += __popc(any);
                }
            }
            ninv = __reduce_add_sync(0xffffffffu, ninv);
            nesc = __reduce_add_sync(0xffffffffu, nesc);
            if (nesc) continue;  // finished by pfa_cds_escape_kernel
            const unsigned long long P = (uint32_t)a.s.pop_n[q] > ninv ? 1ull << codon : 0ull;
            pfa_cds_enqueue(qbuf, qcount, lane, P, 0u, 0u, 0u, q, (uint32_t)site0);
            if (qcount == 32) {
                pfa_cds_flush(qbuf, 32, lane, a.acc_in_smem ? sm_acc : reinterpret_cast<unsigned long long*>(a.out), a.labels, a.s.ns);
                qcount = 0;
                __syncwarp();
            }
        }
        return;
    }
    int nvar = 0, tv = 0, fixed = 0;
    bool fixed_valid = true;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const unsigned ft = (f >> (6 * t)) & 63u;
        if (!pfa_flags_mono(ft)) {
            ++nvar;
            tv = t;
        } else {
            fixed_valid = fixed_valid && (ft & 16u) && !(ft & 32u);
            fixed |= (((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0)) << (2 * (2 - t));
        }
    }
    const int k = MULTI ? a.s.k : 1;
    for (int q = 0; q < k; ++q) {
        const uint32_t* mq = reinterpret_cast<const uint32_t*>(MULTI ? a.s.masks + (int64_t)q * a.s.Wq : a.s.umask);
        const uint32_t nq = (uint32_t)a.s.pop_n[q];
        unsigned long long P = 0ull;
        uint32_t h[3] = {0u, 0u, 0u};
        if (nvar == 1 && fixed_valid) {
            // exactly one site varies, the other two show one valid base: the clean codons are that fixed pair combined with
            // the bases present at the variable site, and only that position can carry a label
            uint32_t c[PFA_NCLASS];
            pfa_coop_counts<HAS_V>(r0 + tv * Wn, r1 + tv * Wn, tv == 0 ? rv[0] : tv == 1 ? rv[1] : rv[2], mq, Wn, lane, c, tv == 0 ? fw[0] : tv == 1 ? fw[1] : fw[2], gcr);
            if (HAS_V && c[PFA_C_ESC]) continue;  // finished by pfa_cds_escape_kernel
            const int shift = 2 * (2 - tv);
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if (c[b]) P |= 1ull << (fixed | (b << shift));
            const uint32_t hv = pfa_site_h32(c, nq);
            h[0] = tv == 0 ? hv : 0u;
            h[1] = tv == 1 ? hv : 0u;
            h[2] = tv == 2 ? hv : 0u;
        } else {
            // general case: class counts of the three columns and the presence mask by peeling distinct codons off each word
            uint32_t cnt[3][PFA_NCLASS];
#pragma unroll
            for (int t = 0; t < 3; ++t)
#pragma unroll
                for (int c = 0; c < PFA_NCLASS; ++c) cnt[t][c] = 0;
            for (int w = lane; w < Wn; w += 32) {
                const uint32_t m = __ldg(mq + w);
                uint32_t live = m;
                uint32_t x[6];
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const uint32_t w0 = r0[t * Wn + w], w1 = r1[t * Wn + w];
                    uint32_t wv = 0xffffffffu;  // words of an unflagged cell were not fetched: all rows valid
                    if (HAS_V && ((fw[t] >> (((unsigned)w * gcr) >> 16)) & 1u)) wv = rv[t][w];
                    const uint32_t vm = HAS_V ? (wv & m) : m;
                    const uint32_t hi = vm & w1, lo = vm & ~w1;
                    cnt[t][PFA_C_T] += __popc(hi & w0);
                    cnt[t][PFA_C_G] += __popc(hi & ~w0);
                    cnt[t][PFA_C_C] += __popc(lo & w0);
                    cnt[t][PFA_C_A] += __popc(lo & ~w0);
                    if (HAS_V) {
                        const uint32_t im = ~wv & m;
                        const uint32_t ihi = im & w1;
                        cnt[t][PFA_C_ESC] += __popc(ihi & w0);
                        cnt[t][PFA_C_Q] += __popc(ihi & ~w0);
                        cnt[t][PFA_C_N] += __popc(im & ~w1 & w0);
                        live &= wv;
                    }
                    x[2 * t] = w1;
                    x[2 * t + 1] = w0;
                }
                while (live) {  // peel one distinct codon per iteration
                    const int r = __ffs(live) - 1;
                    uint32_t match = live;
                    int c = 0;
#pragma unroll
                    for (int t = 0; t < 6; ++t) {
                        const uint32_t bit = (x[t] >> r) & 1u;
                        c = (c << 1) | (int)bit;
                        match &= x[t] ^ (bit - 1u);
                    }
                    P |= 1ull << c;
                    live &= ~match;
                }
            }
            __syncwarp();
#pragma unroll
            for (int t = 0; t < 3; ++t)
#pragma unroll
                for (int c = 0; c < PFA_NCLASS; ++c)
                    if (HAS_V || c < 4) cnt[t][c] = __reduce_add_sync(0xffffffffu, cnt[t][c]);
            P = ((unsigned long long)__reduce_or_sync(0xffffffffu, (uint32_t)(P >> 32)) << 32) | __reduce_or_sync(0xffffffffu, (uint32_t)P);
            if (HAS_V && (cnt[0][PFA_C_ESC] | cnt[1][PFA_C_ESC] | cnt[2][PFA_C_ESC])) continue;  // pfa_cds_escape_kernel
#pragma unroll
            for (int t = 0; t < 3; ++t) h[t] = pfa_site_h32(cnt[t], nq);
        }
        pfa_cds_enqueue(qbuf, qcount, lane, P, h[0], h[1], h[2], q, (uint32_t)site0);
        if (qcount == 32) {
            pfa_cds_flush(qbuf, 32, lane, a.acc_in_smem ? sm_acc : reinterpret_cast<unsigned long long*>(a.out), a.labels, a.s.ns);
            qcount = 0;
            __syncwarp();
        }
    }
}

// pass 1 of a codon column that has flagged cells: mv[t] = the lane's slice of "row of the union AND valid at site t" (the
// site scan's formulation, pfa_site_pass1_valid: everything follows from that one mask per site).  Per site t, six bits at
// 6 t in the layout of pfa_cds_pass1: bits 0-3 the base planes over the VALID rows, bit 4 some row is valid, bit 5 some row is
// not.  Bit 18: a row valid at all three sites exists; bit 19: an escape row (not valid, both base bits set) exists.
template <int LPS, int ITER>
__device__ __forceinline__ unsigned pfa_cds_pass1_valid(const uint4 (&x0)[3][ITER], const uint4 (&x1)[3][ITER], const uint4 (&mv)[3][ITER],
                                                        const uint4 (&um)[ITER], unsigned gmask) {
    unsigned f = 0;
    uint32_t cl = 0, es = 0;
#pragma unroll
    for (int i = 0; i < ITER; ++i)
        cl |= (mv[0][i].x & mv[1][i].x & mv[2][i].x) | (mv[0][i].y & mv[1][i].y & mv[2][i].y) | (mv[0][i].z & mv[1][i].z & mv[2][i].z) |
              (mv[0][i].w & mv[1][i].w & mv[2][i].w);
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        uint32_t o0 = 0, z0 = 0, o1 = 0, z1 = 0, ov = 0, zv = 0;
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            const uint4 m = mv[t][i];
            const uint4 iv = make_uint4(um[i].x ^ m.x, um[i].y ^ m.y, um[i].z ^ m.z, um[i].w ^ m.w);  // rows that are not valid
            zv |= iv.x | iv.y | iv.z | iv.w;
            ov |= m.x | m.y | m.z | m.w;
            es |= (iv.x & x0[t][i].x & x1[t][i].x) | (iv.y & x0[t][i].y & x1[t][i].y) | (iv.z & x0[t][i].z & x1[t][i].z) | (iv.w & x0[t][i].w & x1[t][i].w);
            o0 |= (x0[t][i].x & m.x) | (x0[t][i].y & m.y) | (x0[t][i].z & m.z) | (x0[t][i].w & m.w);
            z0 |= (~x0[t][i].x & m.x) | (~x0[t][i].y & m.y) | (~x0[t][i].z & m.z) | (~x0[t][i].w & m.w);
            o1 |= (x1[t][i].x & m.x) | (x1[t][i].y & m.y) | (x1[t][i].z & m.z) | (x1[t][i].w & m.w);
            z1 |= (~x1[t][i].x & m.x) | (~x1[t][i].y & m.y) | (~x1[t][i].z & m.z) | (~x1[t][i].w & m.w);
        }
        f |= ((o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (ov ? 16u : 0u) | (zv ? 32u : 0u)) << (6 * t);
    }
    f |= (cl ? 1u << 18 : 0u) | (es ? 1u << 19 : 0u);
    return pfa_group_or<LPS>(f, gmask);
}

// One pass of a warp of the TMA kernel over GW codon columns of its slot (whole-warp second pass, LPS >= 4).  V = the block
// carries validity pieces; blocks without a flagged cell run the two-plane instantiation as separate code (see
// pfa_site_tma_pass).
// Columns whose only "variation" is missing data -- at each of the three sites the valid rows show ONE base, no escape row --
// are finished right here: the rows valid at all three sites carry one and the same codon, so as long as every population
// keeps at least one such row the column contributes exactly what a monomorphic column does (stop test, syn-site sum of that
// codon; no labels).  One population: "a clean row exists" is one more OR in pass 1; several: the number of rows that are
// not valid somewhere in the column is compared with the smallest population.  Gaps aligned to codons and runs of N -- the
// usual content of a real CDS alignment -- then cost nothing beyond pass 1.
// bv selects pass 1 (runtime, per block); everything after pass 1 is ONE piece of code for both, with ONE call of `refill` (the
// slot's last pass only, as soon as nothing reads the slot any more): the hot loop has to fit the instruction cache (see
// pfa_site_scan_tma_kernel).
template <int LPS, int ITER, bool HAS_V, bool MULTI, class Refill>
__device__ __forceinline__ void pfa_cds_tma_pass(const PfaCdsArgs& a, const unsigned char* slot, int CPS, unsigned rec, int t0, int64_t blk,
                                                 const uint4 (&um)[ITER], const int (&cell)[ITER], bool bv, bool sparse, unsigned VS, int gcw, int lane,
                                                 int sub, int grp, unsigned gmask, unsigned long long* sm_acc, uint32_t* qbuf, int& qcount,
                                                 unsigned& u_nstops, unsigned& u_missing, unsigned& u_sum3, bool last, Refill&& refill) {
    constexpr int GW = 32 / LPS;
    const int Wq = a.s.Wq, SPS = CPS * 3;
    const int idx = t0 * GW + grp;  // codon column of this group inside the slot
    const int64_t cc = blk * CPS + idx;
    const uint32_t* fa = pfa_slot_flags(slot, (unsigned)SPS, VS, rec);  // flag words of the slot's sites (sparse)
    const unsigned char* gv = reinterpret_cast<const unsigned char*>(a.s.v);
    uint4 x0[3][ITER], x1[3][ITER];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const uint4* q0 = reinterpret_cast<const uint4*>(slot + (size_t)(idx * 3 + t) * rec);
        const uint4* q1 = reinterpret_cast<const uint4*>(slot + (size_t)(SPS + idx * 3 + t) * rec);
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            // unconditional loads: chunks beyond the record (j >= Wq) and columns beyond the end read whatever lies there in
            // the slot (the allocation is padded) -- every use is masked (the masks of those chunks are zero) or dropped
            x0[t][i] = q0[sub + LPS * i];
            x1[t][i] = q1[sub + LPS * i];
        }
    }
    unsigned f, f2 = 0xfffu;  // f2: the base planes over the valid rows, four bits per site ("bases vary" unless pass 1 finds otherwise)
    bool uniform = true, clean = true;
    int codon = 0;
    // the flag words of this column's sites: a column without a flagged cell runs the two-plane pass 1 even inside a block that
    // carries validity pieces (group-uniform branch; in a sparse alignment most columns of a flagged block are clean)
    uint32_t fwg[3] = {0u, 0u, 0u};
    if (HAS_V && bv && cc < a.ncf) {  // a column beyond the end of the shard (last block) has no flag words in the slot
#pragma unroll
        for (int t = 0; t < 3; ++t) fwg[t] = sparse ? fa[idx * 3 + t] : 0xffffffffu;
    }
    if (!(HAS_V && bv) || !(fwg[0] | fwg[1] | fwg[2])) {
        uint4 xv[3][ITER];
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
            for (int i = 0; i < ITER; ++i) xv[t][i] = um[i];
        f = pfa_cds_pass1<LPS, ITER, false>(x0, x1, xv, um, gmask);
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const unsigned ft = (f >> (6 * t)) & 63u;
            uniform = uniform && pfa_flags_bases_mono(ft);
            codon = (codon << 2) | ((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0);
        }
    } else {
        uint4 mv[3][ITER];  // rows of the union that are valid at site t
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const uint4* qv = reinterpret_cast<const uint4*>(
                pfa_slot_vrec(slot, (unsigned)SPS, VS, rec, sparse, idx * 3 + t, gv + (size_t)((cc < a.ncf ? cc : 0) * 3 + t) * rec));
#pragma unroll
            for (int i = 0; i < ITER; ++i) {
                mv[t][i] = um[i];
                if ((fwg[t] >> cell[i]) & 1u) {
                    const uint4 v4 = qv[sub + LPS * i];
                    mv[t][i] = make_uint4(um[i].x & v4.x, um[i].y & v4.y, um[i].z & v4.z, um[i].w & v4.w);
                }
            }
        }
        f = pfa_cds_pass1_valid<LPS, ITER>(x0, x1, mv, um, gmask);
        bool bases_mono = true, some_invalid = false;
        f2 = 0u;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const unsigned ft = (f >> (6 * t)) & 63u;
            bases_mono = bases_mono && pfa_flags_bases_mono(ft);
            some_invalid = some_invalid || (ft & 32u);
            codon = (codon << 2) | ((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0);
            f2 |= (ft & 15u) << (4 * t);
        }
        // at every site the valid rows show ONE base and no row is an escape: as long as every population keeps a row valid at
        // all three sites the column contributes what a monomorphic column does
        uniform = false;
        if (bases_mono && !((f >> 19) & 1u)) {  // group-uniform
            bool every_pop_clean = !some_invalid || ((f >> 18) & 1u);  // one population: a clean row exists
            if (MULTI && some_invalid) {
                uint32_t inv = 0;
#pragma unroll
                for (int i = 0; i < ITER; ++i) {
                    inv += __popc(~(mv[0][i].x & mv[1][i].x & mv[2][i].x) & um[i].x) + __popc(~(mv[0][i].y & mv[1][i].y & mv[2][i].y) & um[i].y) +
                           __popc(~(mv[0][i].z & mv[1][i].z & mv[2][i].z) & um[i].z) + __popc(~(mv[0][i].w & mv[1][i].w & mv[2][i].w) & um[i].w);
                }
                every_pop_clean = pfa_group_add<LPS>(inv, gmask) < (uint32_t)a.min_nq;
            }
            if (every_pop_clean || !MULTI) {
                uniform = true;
                clean = every_pop_clean;  // one population without a clean row: every codon is missing
            }
        }
        f &= 0x3ffffu;  // the whole-warp pass reads the six bits per site
    }
    // variable columns: the whole warp, one at a time, from the slot
    for (unsigned rest = __ballot_sync(0xffffffffu, !uniform && sub == 0 && cc < a.ncf); rest; rest &= rest - 1) {
        const int leader = __ffs(rest) - 1;
        const int vidx = t0 * GW + leader / LPS;
        const unsigned fv = __shfl_sync(0xffffffffu, f, leader), fv2 = __shfl_sync(0xffffffffu, f2, leader);
        const uint32_t* r0 = reinterpret_cast<const uint32_t*>(slot + (size_t)(vidx * 3) * rec);
        const uint32_t* r1 = reinterpret_cast<const uint32_t*>(slot + (size_t)(SPS + vidx * 3) * rec);
        uint32_t fw3[3] = {0u, 0u, 0u};
        if (HAS_V && bv) {
#pragma unroll
            for (int t = 0; t < 3; ++t) fw3[t] = sparse ? fa[vidx * 3 + t] : 0xffffffffu;
        }
        const uint32_t* rv3[3] = {r0, r0, r0};
        if (HAS_V && (fw3[0] | fw3[1] | fw3[2])) {
#pragma unroll
            for (int t = 0; t < 3; ++t)
                rv3[t] = reinterpret_cast<const uint32_t*>(
                    pfa_slot_vrec(slot, (unsigned)SPS, VS, rec, sparse, vidx * 3 + t, gv + (size_t)((blk * CPS + vidx) * 3 + t) * rec));
            pfa_cds_coop<HAS_V, MULTI>(a, (blk * CPS + vidx) * 3, fv, r0, r1, rv3, Wq * 4, lane, sm_acc, qbuf, qcount, fw3, gcw, fv2);
        } else {
            pfa_cds_coop<false, MULTI>(a, (blk * CPS + vidx) * 3, fv, r0, r1, rv3, Wq * 4, lane, sm_acc, qbuf, qcount, fw3, gcw, 0xfffu);
        }
    }
    if (last) refill();
    if (uniform && sub == 0 && cc < a.ncf) {  // the same single codon for every population
        if (clean) {
            u_nstops += (unsigned)((c_stop_mask >> codon) & 1ull);
            u_sum3 += c_syn3[codon];
        } else {
            u_missing += 3;
        }
    }
}

// TMA variant (see pfa_site_scan_tma_kernel): every warp owns a shared-memory slot holding the site records of the codon
// columns of m of its passes (3 * 32/LPS consecutive sites per pass), fed by one cp.async.bulk per plane.  Pass 1 runs per
// group on registers; variable columns (LPS >= 4) are finished by the whole warp one at a time from the slot (pfa_cds_coop).
template <int LPS, int ITER, bool HAS_V, bool MULTI, int NT>
__global__ void __launch_bounds__(NT, 1) pfa_cds_scan_tma_kernel(const PfaCdsArgs a, int m) {
    extern __shared__ __align__(128) unsigned char dyn[];
    constexpr bool COOP = LPS >= 4;  // three site records per column: holding them through pass 2 spills (ptxas), the slot does not
    constexpr int GW = 32 / LPS;        // codon columns per warp pass
    constexpr int NPL = HAS_V ? 3 : 2;  // planes read
    constexpr int NWARP = NT / 32;
    const int Wq = a.s.Wq;
    const unsigned rec = (unsigned)Wq * 16u;  // one site record in one plane
    const int CPS = GW * m;                   // codon columns per slot
    const int SPS = CPS * 3;                  // sites per slot
    const unsigned VS = HAS_V ? (a.s.vs > 0 ? (unsigned)a.s.vs : (unsigned)SPS) : 0u;  // validity records per slot (pfa_slot_issue)
    const unsigned slot_bytes = (unsigned)pfa_slot_bytes(HAS_V, (unsigned)SPS, VS, rec);
    const bool sparse = HAS_V && a.s.vflag != nullptr;  // fetch only the flagged cells of the v plane
    const int gc = a.s.gc, gcw = a.s.gc * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(dyn + (size_t)NWARP * slot_bytes);
    unsigned long long* smem = reinterpret_cast<unsigned long long*>(bars + NWARP);  // [3] uniform + accumulators
    const int nacc = 3 + (a.acc_in_smem ? a.s.k * PFA_CDS_LEN : 0);
    for (int i = threadIdx.x; i < nacc; i += blockDim.x) smem[i] = 0ull;
    if (threadIdx.x == 0) {
        for (int i = 0; i < NWARP; ++i) pfa_mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned long long* sm_acc = smem + 3;

    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sub = lane & (LPS - 1), grp = lane / LPS;
    const unsigned gmask = LPS == 32 ? 0xffffffffu : (((1u << LPS) - 1u) << (lane - sub));
    unsigned u_nstops = 0, u_missing = 0, u_sum3 = 0;
    uint32_t* qbuf = reinterpret_cast<uint32_t*>(smem + nacc) + wib * (PFA_CDS_QFIELDS * 32);  // this warp's queue (COOP)
    int qcount = 0;
    unsigned char* ring = dyn + (size_t)wib * slot_bytes;
    uint64_t* bar = bars + wib;
    const int64_t nw = (int64_t)gridDim.x * NWARP;
    const int64_t nblk = (a.ncf + CPS - 1) / CPS;                    // blocks of CPS consecutive codon columns
    const unsigned char* planes[3] = {reinterpret_cast<const unsigned char*>(a.s.b0), reinterpret_cast<const unsigned char*>(a.s.b1),
                                      reinterpret_cast<const unsigned char*>(a.s.v)};
    uint4 um[ITER];
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        const int j = sub + LPS * i;
        um[i] = j < Wq ? __ldg(a.s.umask + j) : make_uint4(0, 0, 0, 0);
    }
    int cell[ITER];  // the flag bit of each of this lane's chunks
#pragma unroll
    for (int i = 0; i < ITER; ++i) cell[i] = (sub + LPS * i) / gc;
    // block distribution and the one-block-ahead validity flags: see pfa_site_scan_tma_kernel
    PfaClaimer claim;
    const unsigned gw = blockIdx.x * NWARP + wib, nwu = gridDim.x * NWARP;
    const unsigned rounds = (unsigned)(nblk / nwu) * 7u / 8u;  // static rounds of nwu blocks
    unsigned round = 0;
    if (lane == 0) claim.init(a.s.work, (unsigned)nblk - rounds * nwu, nwu);
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
            pfl[u] = (sparse && pend >= 0 && u * 32 + lane < SPS && s < a.ncf * 3) ? __ldg(a.s.vflag + s) : 0u;
        }
    };
    load_flags();
    bool pend_v = HAS_V, cur_v = HAS_V;  // does the block in the slot (being fetched / being scanned) carry validity pieces?
    auto issue_next = [&]() -> int {  // all lanes: fetch `pend` into the warp's slot, then look one block further ahead
        const int blk = pend;
        if (blk >= 0) {
            const int64_t c0 = (int64_t)blk * CPS;
            pend_v = pfa_slot_issue<HAS_V>(ring, bar, planes[0], planes[1], planes[2], sparse, gc, c0 * 3, 3u * (unsigned)min((int64_t)CPS, a.ncf - c0),
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
        for (int t0 = 0; t0 < m; ++t0) {
            if (COOP) {
                pfa_cds_tma_pass<LPS, ITER, HAS_V, MULTI>(a, slot, CPS, rec, t0, blk, um, cell, bv, sparse, VS, gcw, lane, sub, grp, gmask, sm_acc, qbuf, qcount,
                                                          u_nstops, u_missing, u_sum3, t0 == m - 1, refill);
            } else {
                const int idx = t0 * GW + grp;  // codon column of this group inside the slot
                const int64_t cc = blk * CPS + idx;
                uint4 x0[3][ITER], x1[3][ITER], xv[3][ITER];
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const uint4* q0 = reinterpret_cast<const uint4*>(slot + (size_t)(idx * 3 + t) * rec);
                    const uint4* q1 = reinterpret_cast<const uint4*>(slot + (size_t)(CPS * 3 + idx * 3 + t) * rec);
                    const uint4* qv = reinterpret_cast<const uint4*>(slot + (size_t)(2 * CPS * 3 + idx * 3 + t) * rec);
#pragma unroll
                    for (int i = 0; i < ITER; ++i) {
                        const int j = sub + LPS * i;  // unconditional loads, see pfa_cds_tma_pass
                        x0[t][i] = q0[j];
                        x1[t][i] = q1[j];
                        xv[t][i] = HAS_V ? qv[j] : um[i];
                    }
                }
                // pass 1 has consumed every register loaded from the slot: refill it while the rest runs on registers
                const unsigned f = pfa_cds_pass1<LPS, ITER, HAS_V>(x0, x1, xv, um, gmask);
                if (t0 == m - 1) refill();
                if (cc < a.ncf)
                    pfa_cds_finish_regs<LPS, ITER, HAS_V, MULTI>(pfa_cds_view(a), cc * 3, f, x0, x1, xv, um, sub, gmask, Wq, sm_acc, u_nstops, u_missing, u_sum3);
            }
        }
    }
    if (COOP && qcount) pfa_cds_flush(qbuf, qcount, lane, a.acc_in_smem ? sm_acc : reinterpret_cast<unsigned long long*>(a.out), a.labels, a.s.ns);
    if (a.has_partial && blockIdx.x == 0 && threadIdx.x == 0) u_missing += 3;
    for (int off = 16; off; off >>= 1) {
        u_nstops += __shfl_xor_sync(0xffffffffu, u_nstops, off);
        u_missing += __shfl_xor_sync(0xffffffffu, u_missing, off);
        u_sum3 += __shfl_xor_sync(0xffffffffu, u_sum3, off);
    }
    if (lane == 0) {
        if (u_nstops) atomicAdd(&smem[0], (unsigned long long)u_nstops);
        if (u_missing) atomicAdd(&smem[1], (unsigned long long)u_missing);
        if (u_sum3) atomicAdd(&smem[2], (unsigned long long)u_sum3);
    }
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(a.s.work + 1, 1u) == gridDim.x - 1) {  // every CTA has made its last claim
        a.s.work[0] = 0u;
        a.s.work[1] = 0u;
    }
    for (int i = threadIdx.x; i < a.s.k * PFA_CDS_LEN; i += blockDim.x) {
        const int e = i % PFA_CDS_LEN;
        unsigned long long x = a.acc_in_smem ? sm_acc[i] : 0ull;
        if (e == PFA_CDS_NSTOPS) x += smem[0];
        if (e == PFA_CDS_MISSING) x += smem[1];
        if (e == PFA_CDS_SUM3 + 1) x += smem[2];
        if (x) atomicAdd(reinterpret_cast<unsigned long long*>(a.out) + i, x);
    }
    if (a.s.x.world) pfa_xchg_epilogue(a.s.x);
}

// per-site escape statistics of one population: number of distinct escape bytes and the sum of their squared counts
__device__ __forceinline__ void pfa_escape_stats(const unsigned long long* __restrict__ keys, int64_t i0, int64_t i1,
                                                 const uint32_t* __restrict__ mq, unsigned int* hist, int lane,
                                                 uint32_t* distinct_out, unsigned long long* sq_out) {
    for (int b = lane; b < 256; b += 32) hist[b] = 0u;
    __syncwarp();
    for (int64_t i = i0 + lane; i < i1; i += 32) {
        const unsigned long long key = keys[i];
        const uint32_t row = (uint32_t)(key & 0xffffffull);
        if ((mq[row >> 5] >> (row & 31)) & 1u) atomicAdd(&hist[(key >> 24) & 0xffu], 1u);
    }
    __syncwarp();
    uint32_t distinct = 0;
    unsigned long long sq = 0;
    for (int b = lane; b < 256; b += 32) {
        const unsigned long long c = hist[b];
        distinct += c ? 1u : 0u;
        sq += c * c;
    }
    for (int off = 16; off; off >>= 1) {
        distinct += __shfl_xor_sync(0xffffffffu, distinct, off);
        sq += __shfl_xor_sync(0xffffffffu, sq, off);
    }
    __syncwarp();
    *distinct_out = distinct;
    *sq_out = sq;
}

// One warp per codon column that holds an escape symbol (owned by its first exception site).
__global__ void __launch_bounds__(256) pfa_cds_escape_kernel(const PfaCdsArgs a, const unsigned long long* __restrict__ keys,
                                                             int64_t n_exc, const int64_t* __restrict__ heads, int64_t n_heads) {
    __shared__ unsigned int hist[8][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int Wq = a.s.Wq;
    for (int64_t h = wid; h < n_heads; h += nwarps) {
        const int64_t cc = (int64_t)(keys[heads[h]] >> 32) / 3;
        if (cc >= a.ncf) continue;                                                    // trailing partial column
        if (h > 0 && (int64_t)(keys[heads[h - 1]] >> 32) / 3 == cc) continue;        // not the first exception site of cc
        int64_t seg0[3] = {0, 0, 0}, seg1[3] = {0, 0, 0};
        for (int64_t hh = h; hh < n_heads && hh < h + 3; ++hh) {
            const int64_t s = (int64_t)(keys[heads[hh]] >> 32);
            if (s / 3 != cc) break;
            seg0[s % 3] = heads[hh];
            seg1[s % 3] = (hh + 1 < n_heads) ? heads[hh + 1] : n_exc;
        }
        const int64_t site0 = cc * 3;
        for (int q = 0; q < a.s.k; ++q) {
            const uint4* mq = a.s.masks + (int64_t)q * Wq;
            uint32_t cnt[3][PFA_NCLASS];
#pragma unroll
            for (int t = 0; t < 3; ++t)
                pfa_class_counts<true>(a.s.b0 + (site0 + t) * Wq, a.s.b1 + (site0 + t) * Wq, a.s.v + (site0 + t) * Wq, mq, Wq, lane, cnt[t]);
            if (!(cnt[0][PFA_C_ESC] | cnt[1][PFA_C_ESC] | cnt[2][PFA_C_ESC])) continue;  // the main kernel counted it
            uint32_t escd[3] = {0, 0, 0};
            unsigned long long escsq[3] = {0, 0, 0};
            for (int t = 0; t < 3; ++t)
                if (cnt[t][PFA_C_ESC])
                    pfa_escape_stats(keys, seg0[t], seg1[t], reinterpret_cast<const uint32_t*>(mq), hist[wib], lane, &escd[t], &escsq[t]);
            const unsigned long long P = pfa_codon_presence<true>(a.s.b0, a.s.b1, a.s.v, site0, Wq, mq, lane);
            if (lane != 0) continue;
            pfa_cds_contribute(P, cnt, a.s.pop_n[q], escd, escsq, reinterpret_cast<unsigned long long*>(a.out + (int64_t)q * PFA_CDS_LEN),
                               a.labels ? a.labels + (int64_t)q * a.s.ns : nullptr, site0);
        }
    }
}

int pfa_launch_cds_scan(pfa_aln* a, int64_t* d_out, uint8_t* d_labels, pfa_xchg* x) {
    pfa_ctx* ctx = a->ctx;
    if (!ctx->codon_tables_ready) {
        int rc = pfa_upload_codon_tables(ctx);
        if (rc) return rc;
        ctx->codon_tables_ready = true;
    }
    if (a->col_begin % 3 != 0) return pfa_fail(ctx, PFA_ERR_ARG, "cds scan: the shard must start on a codon boundary");
    const bool last = a->col_begin + a->ns == a->L_total;
    if (a->ns % 3 != 0 && !last) return pfa_fail(ctx, PFA_ERR_ARG, "cds scan: only the last shard may end inside a codon");
    const int64_t out_len = (int64_t)PFA_CDS_LEN * a->k;
    // words the site scan left in the exchange's partial buffer (pfa_site_cds_stats_xchg): this scan's vector goes behind them
    // and ONE exchange pushes both; d_out then receives [site vector | codon vector]
    const int64_t carry = x ? pfa_xchg_carry(x) : 0;
    if (x) pfa_xchg_set_carry(x, 0);
    if (carry + out_len > (x ? pfa_xchg_cap(x) : carry + out_len)) return pfa_fail(ctx, PFA_ERR_ARG, "exchange buffer too small for both vectors");
    if (!x) PFA_CUDA(ctx, cudaMemsetAsync(d_out, 0, sizeof(int64_t) * (size_t)out_len, ctx->stream));
    if (d_labels && a->ns) PFA_CUDA(ctx, cudaMemsetAsync(d_labels, 0, (size_t)(a->k * a->ns), ctx->stream));
    if (a->ns == 0 || a->n == 0) return x ? pfa_xchg_launch_only(x, nullptr, carry + out_len, d_out) : PFA_OK;
    PfaCdsArgs args;
    unsigned int* work = nullptr;
    if (int rc = pfa_ctx_work(ctx, &work)) return rc;
    pfa_fill_site_args(a, nullptr, nullptr, &args.s);
    args.out = x ? reinterpret_cast<int64_t*>(pfa_xchg_partial(x)) + carry : d_out;
    args.labels = d_labels;
    args.ncf = a->ns / 3;
    args.has_partial = (a->ns % 3) != 0;
    args.acc_in_smem = (int64_t)a->k * PFA_CDS_LEN * 8 <= 40 * 1024;
    args.min_nq = (int)*std::min_element(a->pop_n.begin(), a->pop_n.end());
    const size_t smem = 8 * (3 + (args.acc_in_smem ? (size_t)a->k * PFA_CDS_LEN : 0));
    int lps = 1;
    while (lps < 32 && (a->Wq + lps - 1) / lps > 2) lps *= 2;
    const int iter = (a->Wq + lps - 1) / lps;
    const bool hv = a->has_invalid != 0, multi = a->k > 1;
    const bool generic = iter > 3;  // lps = 32: records of more than 96 chunks (n > 12,288) stream through one warp per column
    const char* planes = pfa_plane_alloc_name(a->plane_alloc);
    cudaStream_t st = ctx->stream;
    if (x) {  // escape columns first: the scan kernel's last block runs the exchange over the complete shard vector
        if (a->n_exc_sites > 0) {
            int rc = pfa_launch_escape(a, pfa_cds_escape_kernel, args);
            if (rc) return rc;
        }
        int rc = pfa_xchg_fill(x, carry + out_len, d_out, &args.s.x, true);  // the TMA kernels run one CTA per SM
        if (rc) return rc;
    }
    if (!generic) {
        // TMA variant: per-warp shared-memory slots of ~10 KB per plane (three site records per codon column) fed by cp.async.bulk
        const int nt = iter >= 3 ? 256 : 512;
        const int gw = 32 / lps, nwarp = nt / 32;
        const size_t queues = lps >= 4 ? (size_t)nwarp * PFA_CDS_QFIELDS * 32 * sizeof(uint32_t) : 0;  // pfa_cds_flush
        const int m = (int)std::max<int64_t>(1, 10000 / ((int64_t)gw * 3 * a->Wq * 16));
        const PfaTmaShape shape = {3, args.ncf, lps, nt, m, "PFA_CDS_TMA_M", 8, 1, smem + queues, hv};
        PfaTmaPlan p;
        if (int rc = pfa_tma_plan(a, shape, &p)) return rc;
        if (p.sparse_v) args.s.vflag = a->vflag;
        args.s.vs = p.vs;
        const bool found = pfa_for_shape<1, 1, 1, 2, 2, 2, 4, 2, 8, 2, 16, 2, 32, 2, 32, 3>(lps, iter, [&](auto L, auto I) {
            pfa_for_v_multi(hv, multi, [&](auto V, auto M) {
                constexpr int NT = decltype(I)::value >= 3 ? 256 : 512;
                auto kernel = pfa_cds_scan_tma_kernel<decltype(L)::value, decltype(I)::value, decltype(V)::value, decltype(M)::value, NT>;
                cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.dyn);
                kernel<<<p.grid, NT, p.dyn, st>>>(args, p.m);
            });
        });
        if (!found) return pfa_fail(ctx, PFA_ERR_ARG, "cds scan: no TMA kernel for lps=%d iter=%d", lps, iter);
        pfa_note_kernel(ctx, "pfa_cds_scan_tma_kernel<LPS=%d,ITER=%d,HAS_V=%d,MULTI=%d,NT=%d> grid=%u passes_per_slot=%d v_records_per_slot=%d planes=%s",
                        lps, iter, (int)hv, (int)multi, nt, p.grid, p.m, args.s.vs, planes);
        return pfa_scan_done(a, x, true, pfa_cds_escape_kernel, args);
    }
    args.s.x.wide = 0;  // see pfa_launch_site_scan
    const int64_t warps_per_block = PFA_SITE_THREADS / 32;
    const dim3 grid((unsigned)std::min<int64_t>((std::max<int64_t>(args.ncf, 1) + warps_per_block - 1) / warps_per_block, (int64_t)ctx->sm_count * 4));
    if (hv) pfa_cds_scan_kernel<true><<<grid, PFA_SITE_THREADS, smem, st>>>(args);
    else pfa_cds_scan_kernel<false><<<grid, PFA_SITE_THREADS, smem, st>>>(args);
    pfa_note_kernel(ctx, "pfa_cds_scan_kernel<LPS=%d,ITER=%d,HAS_V=%d,MULTI=%d> grid=%u block=%d planes=%s", lps, iter, (int)hv, (int)multi, grid.x,
                    PFA_SITE_THREADS, planes);
    return pfa_scan_done(a, x, true, pfa_cds_escape_kernel, args);
}

// ---- K4b: the codon scan over a batch of small loci (--dir --cds; PolyFastA.py:104 calling :165, :284-315) ----------------
// One warp per tile of PFA_BATCH_CTILE consecutive codon columns of ONE locus (the tile finds its locus by binary search);
// a group of LPS lanes owns a codon column, as in pfa_cds_scan_tma_kernel, and runs the same per-column code
// (pfa_cds_process) on a view of the locus.  Contributions that are the same for every population of the locus -- the
// monomorphic columns -- stay in registers until the end of the tile.
template <int LPS, int ITER>
__global__ void __launch_bounds__(256) pfa_batch_cds_kernel(const PfaBatchArgs a) {
    constexpr int GW = 32 / LPS;
    const int lane = threadIdx.x & 31;
    const int sub = lane & (LPS - 1);
    const unsigned gmask = LPS == 32 ? 0xffffffffu : (((1u << LPS) - 1u) << (lane - sub));
    const long long tile = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (tile >= a.n_ctiles) return;
    const int li = pfa_find_locus(a.ctile_base, a.nloci, tile);
    const PfaLocusDesc d = a.desc[li];
    const int Wq = d.Wq;
    const long long ncf = d.L / 3;
    const long long c_lo = (tile - a.ctile_base[li]) * PFA_BATCH_CTILE, c_hi = min(ncf, c_lo + PFA_BATCH_CTILE);
    const bool hv = a.locus_invalid[li] != 0;
    const uint4* umask = a.masks + d.mask_off + (long long)d.k * Wq;
    PfaCdsView view;
    view.masks = a.masks + d.mask_off;
    view.pop_n = reinterpret_cast<const int64_t*>(a.popn + d.pop_base);
    view.out = reinterpret_cast<int64_t*>(a.cds_out + d.pop_base * PFA_CDS_LEN);
    view.labels = nullptr;
    view.ns = d.L;
    view.k = d.k;
    view.acc_in_smem = 0;
    uint4 um[ITER];
#pragma unroll
    for (int i = 0; i < ITER; ++i) {
        const int j = sub + LPS * i;
        um[i] = j < Wq ? __ldg(umask + j) : make_uint4(0, 0, 0, 0);
    }
    unsigned u_nstops = 0, u_missing = 0, u_sum3 = 0;
    for (long long cc = c_lo + lane / LPS; cc < c_hi; cc += GW) {
        const long long site0 = cc * 3;
        uint4 x0[3][ITER], x1[3][ITER], xv[3][ITER];
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
            for (int i = 0; i < ITER; ++i) {
                const int j = sub + LPS * i;
                x0[t][i] = x1[t][i] = make_uint4(0, 0, 0, 0);
                xv[t][i] = um[i];
                if (j < Wq) {
                    const long long o = d.plane_off + (site0 + t) * Wq + j;
                    x0[t][i] = pfa_ld_stream(a.b0 + o);
                    x1[t][i] = pfa_ld_stream(a.b1 + o);
                    if (hv) xv[t][i] = pfa_ld_stream(a.v + o);
                }
            }
        pfa_cds_process<LPS, ITER, true, true>(view, site0, x0, x1, xv, um, sub, gmask, Wq, nullptr, u_nstops, u_missing, u_sum3);
    }
    __syncwarp();
    if (c_lo == 0 && lane == 0 && d.L % 3 != 0) u_missing += 3;  // the trailing partial column (:305), once per locus
    for (int off = 16; off; off >>= 1) {
        u_nstops += __shfl_xor_sync(0xffffffffu, u_nstops, off);
        u_missing += __shfl_xor_sync(0xffffffffu, u_missing, off);
        u_sum3 += __shfl_xor_sync(0xffffffffu, u_sum3, off);
    }
    for (int q = lane; q < d.k; q += 32) {
        unsigned long long* o = reinterpret_cast<unsigned long long*>(a.cds_out + (d.pop_base + q) * PFA_CDS_LEN);
        if (u_nstops) atomicAdd(&o[PFA_CDS_NSTOPS], (unsigned long long)u_nstops);
        if (u_missing) atomicAdd(&o[PFA_CDS_MISSING], (unsigned long long)u_missing);
        if (u_sum3) atomicAdd(&o[PFA_CDS_SUM3 + 1], (unsigned long long)u_sum3);
    }
}

// codon columns of the batch that hold escape symbols: one warp per column, owned by its first exception site (see
// pfa_cds_escape_kernel); keys carry GLOBAL site indices of the batch
__global__ void __launch_bounds__(256) pfa_batch_cds_escape_kernel(const PfaBatchArgs a, const unsigned long long* __restrict__ keys, long long n_exc,
                                                                   const long long* __restrict__ heads, long long n_heads) {
    __shared__ unsigned int hist[8][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long wid = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long h = wid; h < n_heads; h += nwarps) {
        const long long g = (long long)(keys[heads[h]] >> 32);
        const int li = pfa_find_locus(a.site_base, a.nloci, g);
        const PfaLocusDesc d = a.desc[li];
        const long long s = g - d.site_base, cc = s / 3;
        if (cc >= d.L / 3) continue;  // trailing partial column
        if (h > 0) {                  // not the first exception site of this codon column?
            const long long gp = (long long)(keys[heads[h - 1]] >> 32);
            if (gp >= d.site_base && (gp - d.site_base) / 3 == cc) continue;
        }
        long long seg0[3] = {0, 0, 0}, seg1[3] = {0, 0, 0};
        for (long long hh = h; hh < n_heads && hh < h + 3; ++hh) {
            const long long g2 = (long long)(keys[heads[hh]] >> 32) - d.site_base;
            if (g2 < 0 || g2 >= d.L || g2 / 3 != cc) break;
            seg0[g2 % 3] = heads[hh];
            seg1[g2 % 3] = (hh + 1 < n_heads) ? heads[hh + 1] : n_exc;
        }
        const int Wq = d.Wq;
        const long long site0 = cc * 3;
        const uint4 *p0 = a.b0 + d.plane_off, *p1 = a.b1 + d.plane_off, *pv = a.v + d.plane_off;
        for (int q = 0; q < d.k; ++q) {
            const uint4* mq = a.masks + d.mask_off + (long long)q * Wq;
            uint32_t cnt[3][PFA_NCLASS];
#pragma unroll
            for (int t = 0; t < 3; ++t)
                pfa_class_counts<true>(p0 + (site0 + t) * Wq, p1 + (site0 + t) * Wq, pv + (site0 + t) * Wq, mq, Wq, lane, cnt[t]);
            if (!(cnt[0][PFA_C_ESC] | cnt[1][PFA_C_ESC] | cnt[2][PFA_C_ESC])) continue;  // the main kernel counted it
            uint32_t escd[3] = {0, 0, 0};
            unsigned long long escsq[3] = {0, 0, 0};
            for (int t = 0; t < 3; ++t)
                if (cnt[t][PFA_C_ESC])
                    pfa_escape_stats(keys, seg0[t], seg1[t], reinterpret_cast<const uint32_t*>(mq), hist[wib], lane, &escd[t], &escsq[t]);
            const unsigned long long P = pfa_codon_presence<true>(p0, p1, pv, site0, Wq, mq, lane);
            if (lane != 0) continue;
            pfa_cds_contribute(P, cnt, a.popn[d.pop_base + q], escd, escsq, reinterpret_cast<unsigned long long*>(a.cds_out + (d.pop_base + q) * PFA_CDS_LEN),
                               nullptr, site0);
        }
    }
}

int pfa_launch_batch_cds(pfa_ctx* ctx, const PfaBatchArgs& args, int max_Wq, const unsigned long long* keys, long long n_exc,
                         const long long* heads, long long n_heads) {
    if (!ctx->codon_tables_ready) {
        int rc = pfa_upload_codon_tables(ctx);
        if (rc) return rc;
        ctx->codon_tables_ready = true;
    }
    if (args.n_ctiles > 0) {
        int lps = 1;
        while (lps < 32 && (max_Wq + lps - 1) / lps > 2) lps *= 2;
        const int iter = (max_Wq + lps - 1) / lps;
        const unsigned grid = (unsigned)((args.n_ctiles + 7) / 8);
        cudaStream_t st = ctx->stream;
#define PFA_BC_CASE(L_, I_) \
    if (lps == L_ && iter == I_) pfa_batch_cds_kernel<L_, I_><<<grid, 256, 0, st>>>(args); else
        PFA_BC_CASE(1, 1) PFA_BC_CASE(1, 2) PFA_BC_CASE(2, 2) PFA_BC_CASE(4, 2) PFA_BC_CASE(8, 2) PFA_BC_CASE(16, 2) PFA_BC_CASE(32, 2)
        PFA_BC_CASE(32, 3) PFA_BC_CASE(32, 4)
        return pfa_fail(ctx, PFA_ERR_ARG, "batched codon scan: a locus has too many sequences (Wq=%d); use the single-alignment path", max_Wq);
#undef PFA_BC_CASE
        PFA_LAUNCH_CHECK(ctx);
    }
    if (n_heads > 0) {
        const long long eb = std::min<long long>((n_heads + 7) / 8, (long long)ctx->sm_count * 8);
        pfa_batch_cds_escape_kernel<<<(unsigned)eb, 256, 0, ctx->stream>>>(args, keys, n_exc, heads, n_heads);
        PFA_LAUNCH_CHECK(ctx);
    }
    return PFA_OK;
}

// ---- codon windows (pfa_cds_windows_device): the PFA_CDS_WIN_LEN-word vector of every (population, bin) ------------------
// Bins of g = gcd(W, step) columns as in pfa_windows.cu (g is a multiple of 3 and the shard starts on a codon boundary, so
// every codon column lies in ONE bin).  A bin's vector is what K4 + K2 return for its columns alone:
//   S_s, H_s, S_n, H_n: sums over the bin's sites of K4's labels and K2's per-site H (H of a labelled position is the
//     population's H of the column, :169-170); word PFA_CDS_WIN_S is K2's S (sites with H > 0);
//   nstops, missing, sum3_by_len: functions of the presence mask P of every (codon column, population), as in
//     pfa_cds_contribute.  A column whose three sites are monomorphic over the union and all valid (no flagged cell, or the
//     validity plane says so) shows one codon to every population: its terms stay in registers until the piece ends.
// One warp per piece of at most PFA_CDS_WIN_PIECE sites of a bin (so the number of warps follows ns, not W); every piece adds
// into its bins with one atomic per non-zero word.  bins = [k][PFA_CDS_WIN_LEN][nb], zeroed by the caller.
#define PFA_CDS_WIN_PIECE 96  // sites (32 codon columns) per piece

struct PfaCdsWinArgs {
    PfaSiteArgs s;          // planes, masks, k, Wq, ns, vflag (nullptr: read the validity plane of every column)
    const int64_t* hsite;   // [k][ns] (K2)
    const uint8_t* labels;  // [k][ns] (K4)
    int64_t* bins;
    int64_t c0, g, b0, nb, mpb, ncf;
    int has_partial;  // the shard ends with a partial codon column: +3 missing in its bin
};

__device__ __forceinline__ void pfa_cds_win_add(const PfaCdsWinArgs& a, int q, int w, int64_t j, unsigned long long x) {
    if (x) atomicAdd(reinterpret_cast<unsigned long long*>(a.bins + ((int64_t)q * PFA_CDS_WIN_LEN + w) * a.nb + j), x);
}

__device__ __forceinline__ unsigned long long pfa_warp_sum64(unsigned long long x) {
#pragma unroll
    for (int off = 16; off; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

template <bool HAS_V>
__global__ void __launch_bounds__(256) pfa_cds_window_bins_kernel(const PfaCdsWinArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int Wq = a.s.Wq, k = a.s.k;
    const int64_t ns = a.s.ns, total = a.nb * a.mpb;
    for (int64_t e = warp; e < total; e += nwarps) {  // warp-uniform
        const int64_t j = e / a.mpb, m = e - j * a.mpb;
        const int64_t bs = (a.b0 + j) * a.g + m * PFA_CDS_WIN_PIECE;  // global columns of the piece, clipped to the bin and the shard
        const int64_t lo = max(a.c0, bs) - a.c0, hi = min(min(a.c0 + ns, (a.b0 + j + 1) * a.g), bs + PFA_CDS_WIN_PIECE) - a.c0;
        if (hi <= lo) continue;
        // ---- per-site words ----
        for (int q = 0; q < k; ++q) {
            const int64_t* hq = a.hsite + (int64_t)q * ns;
            const uint8_t* lq = a.labels + (int64_t)q * ns;
            unsigned long long hs = 0, hn = 0, cnt = 0;  // cnt: S at bits 0-15, S_s at 16-31, S_n at 32-47 (a piece < 65,536 sites)
            for (int64_t i = lo + lane; i < hi; i += 32) {
                const int64_t h = hq[i];
                const int l = lq[i];
                cnt += (h != 0 ? 1ull : 0ull) + (l == 1 ? 1ull << 16 : 0ull) + (l == 2 ? 1ull << 32 : 0ull);
                hs += l == 1 ? (unsigned long long)h : 0ull;
                hn += l == 2 ? (unsigned long long)h : 0ull;
            }
            cnt = pfa_warp_sum64(cnt);
            hs = pfa_warp_sum64(hs);
            hn = pfa_warp_sum64(hn);
            if (lane == 0) {
                pfa_cds_win_add(a, q, PFA_CDS_WIN_S, j, cnt & 0xffffull);
                pfa_cds_win_add(a, q, PFA_CDS_SS, j, (cnt >> 16) & 0xffffull);
                pfa_cds_win_add(a, q, PFA_CDS_HS, j, hs);
                pfa_cds_win_add(a, q, PFA_CDS_SN, j, (cnt >> 32) & 0xffffull);
                pfa_cds_win_add(a, q, PFA_CDS_HN, j, hn);
            }
        }
        // ---- codon words ----
        unsigned u_nstops = 0, u_missing = 0, u_sum3 = 0;  // identical for every population
        const int64_t cend = min(hi / 3, a.ncf);
        for (int64_t cc = lo / 3; cc < cend; ++cc) {
            const int64_t site0 = cc * 3;
            bool hv = HAS_V;  // this column's validity plane must be read
            if (HAS_V && a.s.vflag) hv = (__ldg(a.s.vflag + site0) | __ldg(a.s.vflag + site0 + 1) | __ldg(a.s.vflag + site0 + 2)) != 0u;
            unsigned f = 0;  // 6 bits per site as in pfa_cds_scan_kernel: b0 one / zero, b1 one / zero, valid / not valid
            for (int jj = lane; jj < Wq; jj += 32) {
                const uint4 um = __ldg(a.s.umask + jj);
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const uint4 x0 = pfa_ld_stream(a.s.b0 + (site0 + t) * Wq + jj);
                    const uint4 x1 = pfa_ld_stream(a.s.b1 + (site0 + t) * Wq + jj);
                    const uint32_t o0 = (x0.x & um.x) | (x0.y & um.y) | (x0.z & um.z) | (x0.w & um.w);
                    const uint32_t z0 = (~x0.x & um.x) | (~x0.y & um.y) | (~x0.z & um.z) | (~x0.w & um.w);
                    const uint32_t o1 = (x1.x & um.x) | (x1.y & um.y) | (x1.z & um.z) | (x1.w & um.w);
                    const uint32_t z1 = (~x1.x & um.x) | (~x1.y & um.y) | (~x1.z & um.z) | (~x1.w & um.w);
                    uint32_t ov = um.x | um.y | um.z | um.w, zv = 0;
                    if (HAS_V && hv) {
                        const uint4 xv = pfa_ld_stream(a.s.v + (site0 + t) * Wq + jj);
                        ov = (xv.x & um.x) | (xv.y & um.y) | (xv.z & um.z) | (xv.w & um.w);
                        zv = (~xv.x & um.x) | (~xv.y & um.y) | (~xv.z & um.z) | (~xv.w & um.w);
                    }
                    f |= ((o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (ov ? 16u : 0u) | (zv ? 32u : 0u)) << (6 * t);
                }
            }
            f = __reduce_or_sync(0xffffffffu, f);
            bool uniform = true, clean = true;
            int codon = 0;
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                const unsigned ft = (f >> (6 * t)) & 63u;
                const bool mono = ((ft & 3u) != 3u) && ((ft & 12u) != 12u) && ((ft & 48u) != 48u);
                const bool all_escape = (ft & 1u) && (ft & 4u) && !(ft & 16u);
                uniform = uniform && mono && !all_escape;
                clean = clean && (ft & 16u) && !(ft & 32u);
                codon = (codon << 2) | ((ft & 4u) ? 2 : 0) | ((ft & 1u) ? 1 : 0);
            }
            if (uniform) {
                if (clean) {
                    u_nstops += (unsigned)((c_stop_mask >> codon) & 1ull);
                    u_sum3 += c_syn3[codon];
                } else {
                    u_missing += 3;
                }
                continue;
            }
            for (int q = 0; q < k; ++q) {
                const uint4* mq = a.s.masks + (int64_t)q * Wq;
                const unsigned long long P = hv ? pfa_codon_presence<true>(a.s.b0, a.s.b1, a.s.v, site0, Wq, mq, lane)
                                                : pfa_codon_presence<false>(a.s.b0, a.s.b1, a.s.v, site0, Wq, mq, lane);
                if (lane != 0) continue;
                const int len = __popcll(P);
                pfa_cds_win_add(a, q, PFA_CDS_NSTOPS, j, (P & c_stop_mask) ? 1ull : 0ull);
                if (len == 0) {
                    pfa_cds_win_add(a, q, PFA_CDS_MISSING, j, 3ull);
                } else {
                    const unsigned tot3 = (unsigned)__popcll(P & c_syn3_bits[0]) + 2u * (unsigned)__popcll(P & c_syn3_bits[1]) +
                                          4u * (unsigned)__popcll(P & c_syn3_bits[2]);
                    pfa_cds_win_add(a, q, PFA_CDS_SUM3 + len, j, tot3);
                }
            }
        }
        if (a.has_partial && lo <= a.ncf * 3 && a.ncf * 3 < hi) u_missing += 3;  // :305 for the trailing 1-2 sites
        for (int q = lane; q < k; q += 32) {
            pfa_cds_win_add(a, q, PFA_CDS_NSTOPS, j, u_nstops);
            pfa_cds_win_add(a, q, PFA_CDS_MISSING, j, u_missing);
            pfa_cds_win_add(a, q, PFA_CDS_SUM3 + 1, j, u_sum3);
        }
    }
}

int pfa_launch_cds_window_bins(pfa_aln* a, const int64_t* d_hsite, const uint8_t* d_labels, int64_t g, int64_t b0, int64_t nb, int64_t* d_bins) {
    pfa_ctx* ctx = a->ctx;
    if (!ctx->codon_tables_ready) {
        int rc = pfa_upload_codon_tables(ctx);
        if (rc) return rc;
        ctx->codon_tables_ready = true;
    }
    if (a->ns == 0 || nb == 0) return PFA_OK;
    PfaCdsWinArgs args;
    pfa_fill_site_args(a, nullptr, nullptr, &args.s);
    args.s.vflag = a->vflag;  // a column whose three sites have no flagged cell is all valid: its validity records are not read
    args.hsite = d_hsite;
    args.labels = d_labels;
    args.bins = d_bins;
    args.c0 = a->col_begin;
    args.g = g;
    args.b0 = b0;
    args.nb = nb;
    args.mpb = (g + PFA_CDS_WIN_PIECE - 1) / PFA_CDS_WIN_PIECE;
    args.ncf = a->ns / 3;
    args.has_partial = (a->ns % 3) != 0;
    const int64_t warps = nb * args.mpb;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((warps + 7) / 8, (int64_t)ctx->sm_count * 8));
    if (a->has_invalid) pfa_cds_window_bins_kernel<true><<<grid, 256, 0, ctx->stream>>>(args);
    else pfa_cds_window_bins_kernel<false><<<grid, 256, 0, ctx->stream>>>(args);
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}
