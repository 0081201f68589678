// Device helpers shared by the site scan (K2), the escape-site kernel and the codon scan (K4).
#pragma once
#include <algorithm>
#include <type_traits>

#include "pfa_common.cuh"
#include "pfa_xchg.cuh"

#define PFA_SITE_THREADS 256
// packed symbol classes counted with popcounts; the gap class '-' is n_pop minus the others
#define PFA_C_A 0
#define PFA_C_C 1
#define PFA_C_G 2
#define PFA_C_T 3
#define PFA_C_N 4
#define PFA_C_Q 5
#define PFA_C_ESC 6
#define PFA_NCLASS 7

struct PfaSiteArgs {
    const uint4* b0;
    const uint4* b1;
    const uint4* v;
    const uint4* masks;  // [k][Wq]
    const uint4* umask;  // [Wq] union of the populations
    const int64_t* pop_n;    // [k]
    const int64_t* out_off;  // [k] offset of pop q in the int64 result vector ([S, H, sfs...])
    const int64_t* sfs_off;  // [k] offset of pop q's bins in the shared-memory histogram
    int64_t* out;
    uint8_t* isvar;  // optional [k][ns]
    int64_t* hsite;  // optional [k][ns], zero-filled by the launch: H of every variable (site, population), left 0 elsewhere
    int64_t ns;
    int Wq;
    int k;
    int sfs_in_smem;
    int sfs_bins;  // total bins over all populations
    const uint32_t* vflag;  // per-site validity flags (pfa_aln::vflag) or nullptr: fetch the whole v plane
    int gc;                 // chunks per flag bit
    int vs;                 // validity records per slot of the TMA kernels (pfa_slot_issue); 0: as many as sites
    unsigned int* work;  // [2], zero between launches: next block to claim / CTAs done (TMA kernels, pfa_ctx_work)
    PfaXchgDev x;  // x.world > 0: the last block sums `out` over the column shards of all GPUs (pfa_xchg.cuh)
};

// streaming 128-bit load: read-only path, do not allocate in L1 (every byte of the planes is used once)
__device__ __forceinline__ uint4 pfa_ld_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

template <int LPS>
__device__ __forceinline__ unsigned pfa_group_or(unsigned x, unsigned gmask) {
    if (LPS == 32) return __reduce_or_sync(0xffffffffu, x);
#pragma unroll
    for (int off = LPS / 2; off; off >>= 1) x |= __shfl_xor_sync(gmask, x, off);
    return x;
}

template <int LPS>
__device__ __forceinline__ uint32_t pfa_group_add(uint32_t x, unsigned gmask) {
    if (LPS == 32) return __reduce_add_sync(0xffffffffu, x);
#pragma unroll
    for (int off = LPS / 2; off; off >>= 1) x += __shfl_xor_sync(gmask, x, off);
    return x;
}

// counts of the seven packed classes among the rows of one population at one site, summed over the warp
template <bool HAS_V>
__device__ __forceinline__ void pfa_class_counts(const uint4* __restrict__ p0, const uint4* __restrict__ p1,
                                                 const uint4* __restrict__ pv, const uint4* __restrict__ mq, int Wq,
                                                 int lane, uint32_t c[PFA_NCLASS]) {
#pragma unroll
    for (int i = 0; i < PFA_NCLASS; ++i) c[i] = 0;
    for (int j = lane; j < Wq; j += 32) {
        const uint4 m4 = __ldg(mq + j), a4 = __ldg(p0 + j), b4 = __ldg(p1 + j);
        uint4 v4 = m4;
        if (HAS_V) v4 = __ldg(pv + j);
        const uint32_t m[4] = {m4.x, m4.y, m4.z, m4.w}, x0[4] = {a4.x, a4.y, a4.z, a4.w}, x1[4] = {b4.x, b4.y, b4.z, b4.w},
                       xv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t vm = HAS_V ? (xv[w] & m[w]) : m[w];
            const uint32_t hi = vm & x1[w], lo = vm & ~x1[w];
            c[PFA_C_T] += __popc(hi & x0[w]);
            c[PFA_C_G] += __popc(hi & ~x0[w]);
            c[PFA_C_C] += __popc(lo & x0[w]);
            c[PFA_C_A] += __popc(lo & ~x0[w]);
            if (HAS_V) {
                const uint32_t im = ~xv[w] & m[w];
                const uint32_t ihi = im & x1[w];
                c[PFA_C_ESC] += __popc(ihi & x0[w]);
                c[PFA_C_Q] += __popc(ihi & ~x0[w]);
                c[PFA_C_N] += __popc(im & ~x1[w] & x0[w]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < PFA_NCLASS; ++i)
        if (HAS_V || i < 4) c[i] = __reduce_add_sync(0xffffffffu, c[i]);
}

struct PfaSiteResult {
    int isvar;
    int has_escape;
    int sfs_bin;  // -1: fewer than two alleles among A,C,G,T (getsfs is undefined there and skipped)
    unsigned long long h;
};

// (#distinct characters > 1, n^2 - sum_a c_a^2, folded-SFS bin) of one column for one population
// (PolyFastA.py:258, :486-489, :279-281).  esc_distinct / esc_sq describe the escape bytes of the column.
__device__ __forceinline__ PfaSiteResult pfa_site_result(const uint32_t c[PFA_NCLASS], int64_t nq, uint32_t esc_distinct,
                                                          unsigned long long esc_sq) {
    PfaSiteResult r;
    unsigned long long sum = 0, sq = esc_sq;
    int distinct = (int)esc_distinct;
#pragma unroll
    for (int i = 0; i < PFA_NCLASS; ++i) {
        sum += c[i];
        if (i != PFA_C_ESC) {
            sq += (unsigned long long)c[i] * c[i];
            distinct += c[i] ? 1 : 0;
        }
    }
    const unsigned long long gap = (unsigned long long)nq - sum;
    sq += gap * gap;
    distinct += gap ? 1 : 0;
    r.has_escape = c[PFA_C_ESC] != 0;
    r.isvar = distinct > 1;
    r.h = r.isvar ? (unsigned long long)nq * (unsigned long long)nq - sq : 0ull;
    // second largest count among the alleles that are exactly A, C, G, T
    uint32_t m1 = 0, m2 = 0;
    int present = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t x = c[i];
        present += x ? 1 : 0;
        if (x > m1) { m2 = m1; m1 = x; }
        else if (x > m2) m2 = x;
    }
    r.sfs_bin = (present >= 2) ? (int)m2 - 1 : -1;
    return r;
}

// ---- warp-cooperative second pass ----------------------------------------------------------------------------------------
// The first pass of the scan kernels gives a site (or codon column) to a GROUP of LPS lanes; the few variable ones then need
// popcounts per population and scalar bookkeeping.  Done by the owning group alone that work runs with LPS of the 32 lanes
// active (ncu, round 1: 17 active threads per warp in K4, 75 % of all issued instructions).  Here the WHOLE warp takes one
// variable site at a time: lane l counts words l, l + 32, ... of the record (read back from the warp's shared-memory slot),
// REDUX sums the counts, every lane holds the totals and the scalar part runs uniformly (one issue slot per instruction
// whatever the number of active lanes), with the accumulators of population q in the registers of lane q.

// class counts of one population at one site: w0 / w1 / wv point to the site's record in each plane (32-bit words, Wn of
// them), mq to the population's row mask
// fw / gcr: the site's validity flag word and the reciprocal of the 32-bit words per flag bit (pfa_cell_rcp; word w lies in
// cell (w * gcr) >> 16 -- a division here cost 20 instructions per word) -- words of an unflagged cell were not fetched
// (pfa_slot_issue) and count as all valid; fw = ~0, gcr = 0: every word of wv is there
__host__ __device__ __forceinline__ unsigned pfa_cell_rcp(int gcw) { return (65536u + (unsigned)gcw - 1u) / (unsigned)gcw; }  // exact for w * gcw < 65536
template <bool HAS_V>
__device__ __forceinline__ void pfa_coop_counts(const uint32_t* __restrict__ w0, const uint32_t* __restrict__ w1,
                                                const uint32_t* __restrict__ wv, const uint32_t* __restrict__ mq, int Wn, int lane,
                                                uint32_t c[PFA_NCLASS], uint32_t fw = 0xffffffffu, unsigned gcr = 0u) {
#pragma unroll
    for (int i = 0; i < PFA_NCLASS; ++i) c[i] = 0;
    for (int w = lane; w < Wn; w += 32) {
        const uint32_t m = __ldg(mq + w), x0 = w0[w], x1 = w1[w];
        uint32_t xv = 0xffffffffu;
        if (HAS_V && ((fw >> (((unsigned)w * gcr) >> 16)) & 1u)) xv = wv[w];
        const uint32_t vm = HAS_V ? (xv & m) : m;
        const uint32_t hi = vm & x1, lo = vm & ~x1;
        c[PFA_C_T] += __popc(hi & x0);
        c[PFA_C_G] += __popc(hi & ~x0);
        c[PFA_C_C] += __popc(lo & x0);
        c[PFA_C_A] += __popc(lo & ~x0);
        if (HAS_V) {
            const uint32_t im = ~xv & m;
            const uint32_t ihi = im & x1;
            c[PFA_C_ESC] += __popc(ihi & x0);
            c[PFA_C_Q] += __popc(ihi & ~x0);
            c[PFA_C_N] += __popc(im & ~x1 & x0);
        }
    }
#pragma unroll
    for (int i = 0; i < PFA_NCLASS; ++i)
        if (HAS_V || i < 4) c[i] = __reduce_add_sync(0xffffffffu, c[i]);
}

// flags of pass 1 (bit 0/1: plane b0 shows a one / a zero among the rows of the union mask, 2/3: b1, 4/5: v)
__device__ __forceinline__ bool pfa_flags_mono(unsigned f) { return ((f & 3u) != 3u) && ((f & 12u) != 12u) && ((f & 48u) != 48u); }
__device__ __forceinline__ bool pfa_flags_all_escape(unsigned f) { return (f & 1u) && (f & 4u) && !(f & 16u); }
__device__ __forceinline__ bool pfa_flags_bases_mono(unsigned f) { return ((f & 3u) != 3u) && ((f & 12u) != 12u); }

// ---- distribution of the blocks of a scan over the warps of the grid --------------------------------------------------------
// A static split (block b to warp b mod W) left ~7 % of the warp time idle at the end of K4: warps that meet more variable
// columns finish later.  Claiming every block from one counter does not scale (same-address atomics serialise in L2: 5e6
// claims took 10 ms on C4), and even chunked claims cost the memory-bound C4 scan 2 % (a warp-wide broadcast per block;
// measured 3.59 -> 3.66 ms, interleaved chunks 3.68 ms).  So: the first 7/8 of the blocks keep the static split (no
// communication at all), the last 1/8 is handed out dynamically in chunks of consecutive blocks whose size halves from
// phase to phase (guided self-scheduling: with W warps, phase p gives out 4 W chunks of C0 >> p blocks, C0 = blocks / (8 W),
// the last blocks go out one by one); each claim is prefetched one chunk ahead.  PfaClaimer is used by lane 0 of a warp.
struct PfaClaimer {   // block numbers fit 32 bits (a shard has fewer than 2^31 sites)
    unsigned int* ctr;
    unsigned nblk, P, C0, cur, end, pending;
    __device__ __forceinline__ void init(unsigned int* counter, unsigned blocks, unsigned warps) {
        ctr = counter;
        nblk = blocks;
        P = 4u * warps;
        C0 = blocks / (8u * warps);
        if (C0 < 1u) C0 = 1u;
        cur = end = 0u;
        pending = atomicAdd(ctr, 1u);
    }
    __device__ __forceinline__ int next() {  // the next block of this warp, -1 when none is left
        while (cur == end) {
            if (pending == 0xffffffffu) return -1;
            unsigned long long start = 0;
            unsigned c = C0, j = pending;
            while (c > 1u && j >= P) {
                start += (unsigned long long)P * c;
                j -= P;
                c >>= 1;
            }
            start += (unsigned long long)j * c;
            if (start >= nblk) {
                pending = 0xffffffffu;
                return -1;
            }
            cur = (unsigned)start;
            end = start + c < nblk ? (unsigned)start + c : nblk;
            pending = atomicAdd(ctr, 1u);  // needed only when this chunk is used up
        }
        return (int)(cur++);
    }
};

// ---- bulk copies (TMA) into shared memory completing on an mbarrier ------------------------------------------------------
__device__ __forceinline__ uint32_t pfa_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void pfa_mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pfa_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void pfa_mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pfa_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pfa_bulk_load(void* smem_dst, const void* gmem_src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(pfa_smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(pfa_smem_u32(bar))
                 : "memory");
}
// orders this thread's earlier generic-proxy accesses of shared memory before later async-proxy (bulk copy) accesses
__device__ __forceinline__ void pfa_fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void pfa_mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(pfa_smem_u32(bar)),
        "r"(parity)
        : "memory");
}


// ---- fetching one block of consecutive site records into a warp's shared-memory slot ------------------------------------------
// Slot layout: [plane b0: cap_sites records | b1: cap_sites records | v: vs records], then cap_sites flag words and cap_sites
// rank bytes (HAS_V).  Planes b0 and b1 always come whole, one bulk copy each.  The v plane (HAS_V):
//   * vflag == nullptr (dense; vs == cap_sites): whole, a third bulk copy;
//   * sparse: only the flagged cells of each site -- a cell = gc chunks of 16 bytes, one flag bit (pfa_aln::vflag) -- each with
//     its own small bulk copy issued by the lane that holds the site's flag word.  The v area holds the records of the FLAGGED
//     sites side by side (rank = number of flagged sites before it in the block): an alignment with few flagged sites gets a
//     v area of a quarter of a plane (vs = cap_sites / 4, chosen at launch from the density of vflag) and spends the shared
//     memory on more passes per slot instead.  The flag words and ranks go into the slot so that the readers know which
//     words of which record are real (the others count as "all rows valid").  A flagged site beyond the v area (rank >= vs:
//     rare by construction) gets rank 0xff and is read from global memory when it is scanned (pfa_slot_vrec).  With a full v
//     area (vs == cap_sites), when more than a third of the cells of the block are flagged the whole range is fetched after
//     all (flag words all ones, rank = site).
//     (Measured alternatives, 10,000 x 2 Mb at one gap per 10^4 bases, 1.22 ms: the cells chunk by chunk with cp.async /
//     LDGSTS added to the mbarrier with cp.async.mbarrier.arrive 1.32 ms -- three copies and nine scheduling no-ops per cell; the
//     decisions taken before the warp waits for its block and lane 0's bulk copies issued first 1.42 ms.  With every other
//     site flagged the kernel is bound by instruction issue (ncu r2x: 970 instructions per pass of two sites, 60 % issue
//     utilisation with four warps per scheduler), not by bytes or by the copy engine.)
// All copies complete on the slot's mbarrier; lane 0 arms it last with the total byte count (bulk copies that finish before
// the expect_tx only drive the transaction count negative for a moment; the phase cannot complete before lane 0 arrives).
// Called by ALL lanes of the warp; fl[u] = flag word of site 32 u + lane of the block (sparse only).
#define PFA_VF_REGS 2  // sparse validity: at most 32 * PFA_VF_REGS sites per slot
#define PFA_TMA_SMEM_MAX ((size_t)226 * 1024)  // dynamic shared memory of a TMA scan CTA (227 KB per block on sm_100, 128 bytes static)
__host__ __device__ __forceinline__ unsigned pfa_slot_meta_bytes(unsigned cap_sites) {  // flag words + rank bytes
    return ((cap_sites * 4u + 15u) & ~15u) + ((cap_sites + 15u) & ~15u);
}
__host__ __device__ __forceinline__ size_t pfa_slot_bytes(bool has_v, unsigned cap_sites, unsigned vs, unsigned rec) {
    return (size_t)(2u * cap_sites + (has_v ? vs : 0u)) * rec + (has_v ? pfa_slot_meta_bytes(cap_sites) : 0u);
}
__device__ __forceinline__ uint32_t* pfa_slot_flags(unsigned char* slot, unsigned cap_sites, unsigned vs, unsigned rec) {
    return reinterpret_cast<uint32_t*>(slot + (size_t)(2u * cap_sites + vs) * rec);
}
__device__ __forceinline__ const uint32_t* pfa_slot_flags(const unsigned char* slot, unsigned cap_sites, unsigned vs, unsigned rec) {
    return reinterpret_cast<const uint32_t*>(slot + (size_t)(2u * cap_sites + vs) * rec);
}
__device__ __forceinline__ const uint8_t* pfa_slot_ranks(const unsigned char* slot, unsigned cap_sites, unsigned vs, unsigned rec) {
    return slot + (size_t)(2u * cap_sites + vs) * rec + ((cap_sites * 4u + 15u) & ~15u);
}
// the validity record of site idx of the slot (a generic pointer: shared or global memory); gsite = that site's record in the
// v plane in global memory
__device__ __forceinline__ const unsigned char* pfa_slot_vrec(const unsigned char* slot, unsigned cap_sites, unsigned vs, unsigned rec, bool sparse,
                                                              int idx, const unsigned char* gsite) {
    if (!sparse) return slot + (size_t)(2u * cap_sites + (unsigned)idx) * rec;
    const unsigned rk = pfa_slot_ranks(slot, cap_sites, vs, rec)[idx];
    return rk >= vs ? gsite : slot + (size_t)(2u * cap_sites + rk) * rec;  // 0xff: not in the v area
}
// Returns true when the block's v area (or part of it) was fetched; false: the block holds no flagged cell (or the kernel reads no
// validity plane at all) and its sites can be scanned as pure ACGT.
template <bool HAS_V>
__device__ __forceinline__ bool pfa_slot_issue(unsigned char* slot, uint64_t* bar, const unsigned char* p0, const unsigned char* p1,
                                               const unsigned char* pv, bool sparse, int gc, int64_t s0, unsigned nsite, unsigned cap_sites,
                                               unsigned vs, unsigned rec, int Wq, const uint32_t (&fl)[PFA_VF_REGS], int lane) {
    __syncwarp();             // every lane has its last values of the slot's previous contents (consumed by pass 1) ...
    pfa_fence_proxy_async();  // ... and those generic-proxy reads come before the async-proxy writes of the copies
    bool any_flag = HAS_V;
    if (HAS_V && sparse) {
        uint32_t mine = 0;
#pragma unroll
        for (int u = 0; u < PFA_VF_REGS; ++u) mine |= fl[u];
        any_flag = __any_sync(0xffffffffu, mine != 0u);
    }
    if (!(HAS_V && sparse) || !any_flag) {   // whole planes (or no validity piece at all): lane 0 alone
        if (lane == 0) {
            pfa_mbar_expect_tx(bar, (any_flag ? 3u : 2u) * nsite * rec);
            pfa_bulk_load(slot, p0 + (size_t)s0 * rec, nsite * rec, bar);
            pfa_bulk_load(slot + (size_t)cap_sites * rec, p1 + (size_t)s0 * rec, nsite * rec, bar);
            if (any_flag) pfa_bulk_load(slot + (size_t)2 * cap_sites * rec, pv + (size_t)s0 * rec, nsite * rec, bar);
        }
        return any_flag;
    }
    unsigned vbytes = HAS_V ? nsite * rec : 0u;
    bool whole_v = HAS_V;
    if (HAS_V && sparse) {
        uint32_t* fa = pfa_slot_flags(slot, cap_sites, vs, rec);
        uint8_t* ra = const_cast<uint8_t*>(pfa_slot_ranks(slot, cap_sites, vs, rec));
        unsigned cells = 0;
#pragma unroll
        for (int u = 0; u < PFA_VF_REGS; ++u)
            if ((unsigned)(u * 32) < nsite && (unsigned)(u * 32 + lane) < nsite) cells += __popc(fl[u]);
        cells = __reduce_add_sync(0xffffffffu, cells);
        const unsigned ncell = (unsigned)((Wq + gc - 1) / gc);
        whole_v = vs == cap_sites && cells * 3u > nsite * ncell;
        unsigned bytes = 0, base = 0;
#pragma unroll
        for (int u = 0; u < PFA_VF_REGS; ++u) {
            const unsigned si = (unsigned)(u * 32 + lane);
            const bool live = (unsigned)(u * 32) < nsite && si < nsite;
            const unsigned flagged = __ballot_sync(0xffffffffu, live && fl[u] != 0u);
            const unsigned rank = base + (unsigned)__popc(flagged & ((1u << lane) - 1u));
            base += (unsigned)__popc(flagged);
            if (live) {
                const bool resident = whole_v || (fl[u] != 0u && rank < vs);
                fa[si] = whole_v ? 0xffffffffu : fl[u];
                ra[si] = (uint8_t)(whole_v ? si : resident ? rank : 0xffu);
                if (!whole_v && resident)
                    for (uint32_t w = fl[u]; w; w &= w - 1) {
                        const int c0 = (__ffs(w) - 1) * gc;
                        const unsigned len = (unsigned)min(gc, Wq - c0) * 16u;
                        pfa_bulk_load(slot + (size_t)(2u * cap_sites + rank) * rec + (size_t)c0 * 16u, pv + (size_t)(s0 + si) * rec + (size_t)c0 * 16u, len, bar);
                        bytes += len;
                    }
            }
        }
        bytes = __reduce_add_sync(0xffffffffu, bytes);
        if (!whole_v) vbytes = bytes;
    }
    __syncwarp();
    if (lane == 0) {
        pfa_mbar_expect_tx(bar, 2u * nsite * rec + vbytes);
        pfa_bulk_load(slot, p0 + (size_t)s0 * rec, nsite * rec, bar);
        pfa_bulk_load(slot + (size_t)cap_sites * rec, p1 + (size_t)s0 * rec, nsite * rec, bar);
        if (whole_v) pfa_bulk_load(slot + (size_t)2 * cap_sites * rec, pv + (size_t)s0 * rec, nsite * rec, bar);
    }
    return true;
}

void pfa_fill_site_args(const pfa_aln* a, int64_t* d_out, uint8_t* d_isvar, PfaSiteArgs* args, int64_t* d_hsite = nullptr);
int pfa_aln_flagged_sites(pfa_aln* a, int64_t* out);

// ---- launch plan of the TMA scans (K2, K4) -----------------------------------------------------------------------------------
// what the site scan (a unit = one site record) and the codon scan (a unit = a codon column, three site records) tell the planner
struct PfaTmaShape {
    int recs;           // site records per unit; a slot's validity area holds at least one unit
    int64_t units;      // units in the shard
    int lps;            // lanes per unit
    int nt;             // threads per CTA
    int m;              // passes per slot, unless m_env is set
    const char* m_env;  // the variable that overrides m
    int v_div_max;      // sparse validity: the v area is 1/d of the slot's records, d = the largest power of two <= v_div_max
                        // with at most 1/d^2 of the sites flagged
    int m_raise;        // a v area below a whole slot raises m to m + ceil(m * m_raise / 2) (no m_env)
    size_t smem;        // shared memory beyond the slots and their mbarriers: accumulators, queues
    bool has_v;         // the scan reads the validity plane (pfa_aln::has_invalid)
};
struct PfaTmaPlan {
    bool sparse_v;          // fetch only the flagged cells of the v plane (PfaSiteArgs::vflag)
    int64_t flagged_sites;  // sites with a flagged cell (sparse_v)
    int v_div;              // v area = records per slot / v_div
    int m;                  // passes per slot
    int vs;                 // validity records per slot (PfaSiteArgs::vs)
    size_t dyn;             // dynamic shared memory of a CTA
    unsigned grid;          // CTAs: at most one per SM
};
int pfa_tma_plan(pfa_aln* a, const PfaTmaShape& s, PfaTmaPlan* p);

// f(integral_constant<int, L>, integral_constant<int, I>) for the pair (L, I) of the list that equals (lps, iter); false: none
template <class F>
bool pfa_for_shape(int, int, F&&) {
    return false;
}
template <int L, int I, int... Rest, class F>
bool pfa_for_shape(int lps, int iter, F&& f) {
    if (lps == L && iter == I) {
        f(std::integral_constant<int, L>{}, std::integral_constant<int, I>{});
        return true;
    }
    return pfa_for_shape<Rest...>(lps, iter, f);
}

// f(integral_constant<bool, HAS_V>, integral_constant<bool, MULTI>) for the runtime pair
template <class F>
void pfa_for_v_multi(bool has_v, bool multi, F&& f) {
    using T = std::true_type;
    using N = std::false_type;
    if (has_v && multi) f(T{}, T{});
    else if (has_v) f(T{}, N{});
    else if (multi) f(N{}, T{});
    else f(N{}, N{});
}

// one warp per site (K2) or codon column (K4) that holds an escape symbol
template <class Args>
int pfa_launch_escape(pfa_aln* a, void (*kernel)(Args, const unsigned long long*, int64_t, const int64_t*, int64_t), const Args& args) {
    pfa_ctx* ctx = a->ctx;
    const int64_t eb = std::min<int64_t>((a->n_exc_sites + 7) / 8, (int64_t)ctx->sm_count * 8);
    kernel<<<(unsigned)eb, 256, 0, ctx->stream>>>(args, a->exc_keys, a->n_exc, a->exc_heads, a->n_exc_sites);
    PFA_LAUNCH_CHECK(ctx);
    return PFA_OK;
}

// after the scan kernel: check its launch, then commit the exchange it feeds (x, commit) -- whose escape kernel went first, so
// that the scan's last block sees the complete shard vector -- or, without an exchange, run the escape kernel now
template <class Args>
int pfa_scan_done(pfa_aln* a, pfa_xchg* x, bool commit, void (*escape)(Args, const unsigned long long*, int64_t, const int64_t*, int64_t),
                  const Args& args) {
    PFA_LAUNCH_CHECK(a->ctx);
    if (x && commit) pfa_xchg_commit(x);
    if (!x && a->n_exc_sites > 0) return pfa_launch_escape(a, escape, args);
    return PFA_OK;
}
