// Shared declarations of the polyfasta_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/polyfasta_b200.h"

#define PFA_SM_COUNT_FALLBACK 148

// where an alignment's planes live (pfa_aln_plane_alloc)
enum { PFA_PLANES_POOL = 0, PFA_PLANES_VMM = 1, PFA_PLANES_COMPRESSIBLE = 2 };

// a virtual-memory range mapped onto one physical allocation (cuMemCreate): `want` is the kind asked for, `kind` the kind
// granted (a device without compressible memory grants PFA_PLANES_VMM)
struct pfa_vmm_range {
    void* ptr = nullptr;
    size_t size = 0;
    unsigned long long handle = 0;  // CUmemGenericAllocationHandle
    int want = 0, kind = 0;
};

// ---- handles ----------------------------------------------------------------------------------------
struct pfa_ctx {
    int device = 0;
    int sm_count = PFA_SM_COUNT_FALLBACK;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;  // own_stream or a caller-owned stream
    std::string err;
    std::string last_kernel;  // the scan kernel of the last K2 / K4 launch, as instantiated (pfa_ctx_last_kernel)
    std::atomic<int64_t> launches{0};  // kernels launched (the packed ingest lane launches from its own thread)
    // small pinned + device scratch for finalisation and synchronous result copies
    void* h_scratch = nullptr;
    void* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    // upload pipeline: copy stream + events, created once per context
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[3] = {}, ev_encoded[3] = {}, ev_ready = nullptr;
    // hybrid ingest (pfa_ingest.cu): encode stream of the raw lane, copy + encode stream of the packed lane, one event per
    // packed staging slot, pinned staging for the host-packed chunks (kept between uploads)
    cudaStream_t enc_stream = nullptr, pack_stream = nullptr;
    cudaEvent_t ev_slot[6] = {}, ev_slot_copied[6] = {}, ev_join[2] = {nullptr, nullptr};
    void* pack_pinned = nullptr;
    size_t pack_pinned_bytes = 0;
    void* raw_pinned = nullptr;  // bounce buffers for text chunks of a pageable source
    size_t raw_pinned_bytes = 0;
    unsigned int* d_work = nullptr;  // block-claim counters of the TMA scan kernels (zero between launches)
    bool codon_tables_ready = false;  // constant-memory tables of K4 uploaded (first codon scan)
    int host_threads = 0;  // host threads the ingest may use; 0 = PFA_HOST_THREADS or all hardware threads
    int64_t ingest_stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // last upload: chunks sent as text, chunks packed on the host, dirty chunks, threads, H2D bytes as text, H2D bytes packed, packed chunks that carried a validity bitmap
    // the VMM range of the planes of the last freed alignment: the next alignment that fits takes it over (mapping tens of GB
    // costs milliseconds).  Unmapped only after a synchronise of the stream (pfa_ctx_trim, pfa_ctx_destroy, a larger request).
    pfa_vmm_range plane_cache;
};

struct pfa_aln {
    pfa_ctx* ctx = nullptr;
    int64_t n = 0;          // rows
    int64_t L_total = 0;    // sites of the whole alignment
    int64_t col_begin = 0;  // first global column of this shard
    int64_t ns = 0;         // sites in this shard
    int Wq = 0;             // uint4 per site per plane = ceil(n/128)
    uint4* planes = nullptr;  // one allocation: b0 | b1 | v
    int plane_alloc = PFA_PLANES_POOL;  // where `planes` came from
    pfa_vmm_range plane_vmm;  // the range behind `planes` unless they came from the pool
    uint4 *b0 = nullptr, *b1 = nullptr, *v = nullptr;
    size_t plane_bytes = 0;  // bytes of ONE plane (ns*Wq*16, padded to 256)
    int has_invalid = 0;  // bit 0: a row shows a symbol outside ACGT somewhere; bit 1: forced (benchmarks: read the v plane everywhere)
    // validity flags, one 32-bit word per site: bit c is set when one of the chunks [c*gc, (c+1)*gc) of the site's v record holds
    // a zero among the real rows.  Written by the encoders; the TMA scans fetch only flagged pieces of the v plane.
    uint32_t* vflag = nullptr;
    int64_t vflag_sites = -1;  // sites with a flag word != 0 (-1: not counted yet; pfa_aln_flagged_sites)
    int gc = 1;  // chunks (16 bytes = 128 rows) per flag bit: ceil(Wq / 32)
    // exception list: sorted keys (site:32 | byte:8 | row:24), heads = first index of every distinct site
    unsigned long long* exc_keys = nullptr;
    int64_t n_exc = 0;
    int64_t* exc_heads = nullptr;
    int64_t n_exc_sites = 0;
    // populations
    int k = 1;
    uint4* d_masks = nullptr;  // [k][Wq]
    uint4* d_union = nullptr;  // [Wq]
    int64_t* d_pop_n = nullptr;
    int64_t* d_site_off = nullptr;
    std::vector<int64_t> pop_n;
    std::vector<int64_t> site_off;  // offsets into the site result vector, size k+1
    // the sites of this shard at which two of the n rows differ in the planes, ascending (built lazily, pfa_var_sites_ensure;
    // dropped with rowmajor by every writer of the planes): the sites the TMA site scan, the divergence scan and the row-major
    // planes visit.  n_var_sites: their number, -1 while the list is not built.
    int64_t* var_sites = nullptr;
    int64_t n_var_sites = -1;
    // row-major copy of the listed sites for the pairwise kernel and the haplotype classes (built lazily, pfa_rowmajor_ensure):
    // [plane][n][Wl] uint32, Wl = ceil(n_var_sites/32) padded to 4
    uint32_t* rowmajor = nullptr;
    int rowmajor_planes = 0;  // 2: pure-ACGT shard (b0, b1), 3: with the validity plane
    int64_t Wl = 0;
    // the exception list by row (built lazily, pfa_haplotypes.cu): keys (row:24 | site:32 | byte:8) sorted, and [n + 1] offsets:
    // row r's entries are exc_rows[exc_row_off[r] .. exc_row_off[r + 1])
    unsigned long long* exc_rows = nullptr;
    int64_t* exc_row_off = nullptr;
};

// ---- error plumbing ----------------------------------------------------------------------------------
int pfa_fail(pfa_ctx* ctx, int code, const char* fmt, ...);
void pfa_set_global_error(const char* fmt, ...);
void pfa_note_kernel(pfa_ctx* ctx, const char* fmt, ...);
static inline const char* pfa_plane_alloc_name(int kind) {
    return kind == PFA_PLANES_COMPRESSIBLE ? "compressible" : kind == PFA_PLANES_VMM ? "vmm" : "pool";
}

#define PFA_CUDA(ctx, call)                                                                       \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return pfa_fail((ctx), PFA_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                            __FILE__, __LINE__);                                                  \
    } while (0)

#define PFA_LAUNCH_CHECK(ctx)                                                                     \
    do {                                                                                          \
        (ctx)->launches++;                                                                        \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess)                                                                   \
            return pfa_fail((ctx), PFA_ERR_CUDA, "kernel launch failed: %s (%s:%d)",              \
                            cudaGetErrorString(e__), __FILE__, __LINE__);                         \
    } while (0)

// ---- internal entry points implemented in the .cu files -----------------------------------------------
int pfa_encode_chunk(pfa_aln* a, const uint8_t* d_text, int64_t ldt, int64_t cols, int64_t site0,
                     unsigned long long* d_exc_count, int64_t exc_cap, int* d_has_invalid, cudaStream_t st = nullptr);
int pfa_finish_exceptions(pfa_aln* a, int64_t count);
int pfa_sort_exceptions(pfa_ctx* ctx, unsigned long long** keys, int64_t count, int64_t** heads, int64_t* n_heads);
int pfa_launch_finalize(pfa_ctx* ctx, const pfa_final_in* d_in, pfa_final_out* d_out, int count);
int pfa_synth_fill(pfa_aln* a, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm);
struct pfa_xchg;
struct PfaXchgDev;
// x != nullptr: fused with the sum over the column shards of all ranks (pfa_xchg.cu); d_out receives the reduced vector
// defer (with x): the shard's vector stays in the exchange's partial buffer and travels with the next exchange (the codon scan's)
// d_hsite (optional): int64 [k][ns], H of every variable (site, population), 0 elsewhere (pfa_site_stats_hsite_device)
int pfa_launch_site_scan(pfa_aln* a, int64_t* d_out, uint8_t* d_isvar, pfa_xchg* x = nullptr, bool defer = false,
                         int64_t* d_hsite = nullptr);
// windows of this shard (pfa_windows.cu) for `rows` rows of per-site values d_persite [rows][ns]: d_counts [rows][nwin][2] =
// (non-zero sites, sum); the site scan's per-site H gives (S, H) per population, the divergence scan's Dxy_site per pair
int pfa_launch_row_windows(pfa_aln* a, int rows, const int64_t* d_persite, int64_t window, int64_t step, int64_t* d_counts);
// a->var_sites and a->n_var_sites, built once per alignment (pfa_pairwise.cu)
cudaError_t pfa_var_sites_ensure(pfa_aln* a);
// drops what was derived from the planes (the site list, the row-major planes): every writer of the planes after construction
void pfa_aln_planes_changed(pfa_aln* a);
int pfa_launch_cds_scan(pfa_aln* a, int64_t* d_out, uint8_t* d_labels, pfa_xchg* x = nullptr);
// codon windows: bins [k][PFA_CDS_WIN_LEN][nb] (zeroed) of this shard from K2's per-site H and K4's labels (pfa_codon.cu), and
// the window vectors [k][nwin][PFA_CDS_WIN_LEN] from them (pfa_windows.cu)
int pfa_launch_cds_window_bins(pfa_aln* a, const int64_t* d_hsite, const uint8_t* d_labels, int64_t g, int64_t b0, int64_t nb, int64_t* d_bins);
int pfa_launch_cds_windows(pfa_aln* a, const int64_t* d_hsite, const uint8_t* d_labels, int64_t window, int64_t step, int64_t* d_counts);
int pfa_xchg_fill(pfa_xchg* x, int64_t len, int64_t* d_out, PfaXchgDev* dev, bool coresident = false);
unsigned long long* pfa_xchg_partial(pfa_xchg* x);
void pfa_xchg_commit(pfa_xchg* x);
int64_t pfa_xchg_carry(const pfa_xchg* x);
void pfa_xchg_set_carry(pfa_xchg* x, int64_t words);
int64_t pfa_xchg_cap(const pfa_xchg* x);
int pfa_xchg_launch_only(pfa_xchg* x, const int64_t* d_src, int64_t len, int64_t* d_out);
int pfa_launch_pairwise(pfa_aln* a, int64_t* d_out, int32_t* d_matrix);
// K3's step 1 (pfa_pairwise.cu): a->rowmajor, built once per alignment and number of planes
cudaError_t pfa_rowmajor_ensure(pfa_aln* a);
int pfa_upload_codon_tables(pfa_ctx* ctx);
int pfa_ctx_work(pfa_ctx* ctx, unsigned int** out);
int pfa_aln_alloc(pfa_ctx* ctx, int64_t n, int64_t L, int64_t col_begin, int64_t col_end, pfa_aln** out);
int pfa_aln_default_pop(pfa_aln* a);
// upload + encode of columns [col_begin, col_end) of a text matrix (pfa_ingest.cu); `dev`: the matrix is in device memory
// row_off (host sources only, optional): row r starts at text + row_off[r] instead of text + r * ld; wrap_w / wrap_gap
// (optional, with row_off): row r is wrapped over lines of wrap_w[r] bytes every wrap_w[r] + wrap_gap[r] bytes (0: contiguous)
int pfa_aln_from_text(pfa_ctx* ctx, const uint8_t* text, bool dev, int64_t n, int64_t L, int64_t ld, int64_t col_begin,
                      int64_t col_end, pfa_aln** out, const int64_t* row_off = nullptr, const int32_t* wrap_w = nullptr,
                      const int32_t* wrap_gap = nullptr);
int pfa_encode_packed_chunk(pfa_aln* a, const uint8_t* d_packed, int64_t ldp, const uint8_t* d_valid, int64_t ldv, int direct,
                            int64_t cols, int64_t site0, int* d_has_invalid, cudaStream_t st);

// Device memory comes from the device's stream-ordered pool (release threshold = keep): allocating and freeing the planes
// of one alignment after another (--dir mode, benchmark loops) reuses the same blocks without synchronising the device.
template <typename T>
static inline cudaError_t pfa_dmalloc(pfa_ctx* ctx, T** p, size_t bytes) {
    return cudaMallocAsync(reinterpret_cast<void**>(p), bytes ? bytes : 16, ctx->stream);
}
static inline void pfa_dfree(pfa_ctx* ctx, void* p) {
    if (p) cudaFreeAsync(p, ctx->stream);
}

static inline int64_t pfa_round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
