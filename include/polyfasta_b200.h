/* polyfasta_b200 -- C ABI of the B200-native PolyFastA hot path.
 *
 * The reference (PolyFastA.py, pure Python) has no FFI; its seams are the function calls inside
 * print_result.no_header (PolyFastA.py:149,165,172-173,191).  Each entry point below names the reference
 * code it replaces.  Plain pointers and sizes only; every call returns an int status (0 = PFA_OK); no
 * C++ exception crosses the boundary; the library owns all device and pinned memory behind opaque
 * handles; there is NO CPU fallback -- without a CUDA device every compute entry point fails with
 * PFA_ERR_CUDA.  Calls on one handle are not re-entrant.
 *
 * Device layout (see DESIGN.md): three site-major bit-planes over rows, b0 / b1 / v, each
 * uint4[sites][Wq] with Wq = ceil(n/128) (rounded up to an even number from 16 on: whole 32-byte sectors).  v=1: A,C,G,T = b1b0 00,01,10,11.  v=0: '-','N','?' = 00,01,10
 * and 11 = "escape" (any other byte; its identity is kept in a sorted exception list).
 */
#ifndef POLYFASTA_B200_H
#define POLYFASTA_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PFA_OK 0
#define PFA_ERR_CUDA 1      /* CUDA runtime error or no device; text via pfa_last_error */
#define PFA_ERR_ARG 2
#define PFA_ERR_NOT_FASTA 3 /* PolyFastA.py:246-248 "# file ... is not FASTA!" */
#define PFA_ERR_RAGGED 4    /* PolyFastA.py:112,135-140 "# Sequences do not have the same length" */
#define PFA_ERR_IO 5
#define PFA_ERR_NOMEM 6
#define PFA_ERR_NON_ASCII 7 /* bytes >= 0x80 in sequence lines: len() in code points != bytes; unsupported */

typedef struct pfa_ctx pfa_ctx;     /* one CUDA device + stream + scratch */
typedef struct pfa_fasta pfa_fasta; /* one parsed FASTA file on the host  */
typedef struct pfa_aln pfa_aln;     /* one alignment (or column shard of one) resident in HBM */

int pfa_version(void);
int pfa_device_count(void);
const char* pfa_global_error(void); /* error text of the last failed call that had no ctx */

/* ---- context ------------------------------------------------------------------------------------ */
int pfa_ctx_create(int device, pfa_ctx** out);
int pfa_ctx_destroy(pfa_ctx* ctx);
const char* pfa_last_error(const pfa_ctx* ctx);
int pfa_ctx_sync(pfa_ctx* ctx);
/* device memory freed by the library stays in the device's stream-ordered pool for reuse, and the planes of the last freed
 * alignment stay mapped for the next one; this synchronises the ctx's stream and returns both to the driver */
int pfa_ctx_trim(pfa_ctx* ctx);
/* run the library's work for this ctx on a caller-owned stream (cudaStream_t as void*; e.g. torch's
 * current stream) so that a collective enqueued by the caller is ordered after the kernels. NULL restores
 * the ctx's own stream. */
int pfa_ctx_set_stream(pfa_ctx* ctx, void* cuda_stream);
/* host threads the ingest may use to pack column chunks (0 = the PFA_HOST_THREADS environment variable, else all hardware
 * threads); with several ranks on one box give every rank its share */
int pfa_ctx_set_host_threads(pfa_ctx* ctx, int threads);
/* the last upload of this ctx: out[0] column chunks shipped as text (K1), out[1] chunks packed 4 bases/byte on the host
 * (pfa_encode_packed_kernel), out[2] chunks the packer found dirty (non-ACGT) and handed back, out[3] host threads,
 * out[4] bytes copied host->device as text, out[5] bytes copied host->device packed, out[6] packed chunks that carried a
 * validity bitmap (gaps / N / ?; needs AVX-512 VBMI on the host, else such chunks count as dirty), out[7] reserved */
int pfa_ctx_ingest_stats(const pfa_ctx* ctx, int64_t out[8]);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
int64_t pfa_ctx_launch_count(const pfa_ctx* ctx);
/* the site / codon scan kernel of the last K2 / K4 launch on this context as it was instantiated and launched (benchmarks) */
const char* pfa_ctx_last_kernel(const pfa_ctx* ctx);

/* ---- ingest: replaces readfasta (PolyFastA.py:227-250) -------------------------------------------- */
/* Parsing semantics of the reference: a line whose first byte is '>' starts a record, header = rest of
 * the line right-stripped; a repeated header restarts that record in place; lines before the first
 * non-empty header are dropped; sequence lines are right-stripped (upper-casing happens in the encoder
 * and in pfa_fasta_copy_row).  Returns PFA_ERR_NOT_FASTA when the reference would. */
int pfa_fasta_parse_file(const char* path, pfa_fasta** out);
int pfa_fasta_parse_buffer(const void* buf, size_t len, pfa_fasta** out);
void pfa_fasta_free(pfa_fasta* f);
int64_t pfa_fasta_nseq(const pfa_fasta* f);
int64_t pfa_fasta_seqlen(const pfa_fasta* f); /* common length, or -1 when rows differ in length */
int64_t pfa_fasta_row_len(const pfa_fasta* f, int64_t row);
const char* pfa_fasta_header(const pfa_fasta* f, int64_t row, int64_t* len); /* not NUL-terminated */
/* upper-cased copy of one row into caller memory (cap >= row_len) */
int pfa_fasta_copy_row(const pfa_fasta* f, int64_t row, uint8_t* dst, int64_t cap);

/* host packer of the ingest, exposed for tests: cols bases of one text row -> ceil(cols/4) bytes, base j of a byte at bits
 * 2j..2j+1, code = (byte >> 1) & 3 (A 0, C 1, T 2, G 3, either case).  Returns 1 when the row holds any other byte (such
 * column chunks are uploaded as text and encoded by K1 instead), 0 when clean, < 0 on bad arguments / unsupported variant.
 * variant: 0 = best for this CPU, 1 = scalar, 2 = AVX2, 3 = AVX-512BW. */
int pfa_host_pack2(const uint8_t* src, int64_t cols, uint8_t* dst, int variant);
/* the packer with a validity bitmap (gaps, N and ? travel packed too): codes A0 C1 G2 T3 / '-'0 'N'1 '?'2 into
 * codes[ceil(cols/4)], one validity bit per base into valid[ceil(cols/8)].  Returns bit 0 = the row holds '-', 'N' or '?',
 * bit 1 = it holds any other byte (dirty); < 0 on bad arguments / unsupported variant (0 best, 1 scalar, 4 AVX-512 VBMI). */
int pfa_host_pack3(const uint8_t* src, int64_t cols, uint8_t* codes, uint8_t* valid, int variant);
/* a whole matrix text[row*ld + col] -> dst[row*ldp + col/4] with `threads` host threads (0 = all); returns the dirty rows */
int64_t pfa_host_pack2_rows(const uint8_t* text, int64_t n, int64_t cols, int64_t ld, uint8_t* dst, int64_t ldp, int threads);

/* ---- alignment upload: host text -> packed planes in HBM (kernel K1) ------------------------------- */
/* columns [col_begin, col_end) of a parsed file (the column shard of this GPU) */
int pfa_aln_from_fasta(pfa_ctx* ctx, const pfa_fasta* f, int64_t col_begin, int64_t col_end, pfa_aln** out);
/* same from a raw row-major byte matrix text[row*ld + col] in host memory (pinned or pageable) */
int pfa_aln_from_rows(pfa_ctx* ctx, const uint8_t* text, int64_t n, int64_t L, int64_t ld,
                      int64_t col_begin, int64_t col_end, pfa_aln** out);
/* same from a byte matrix already in device memory */
int pfa_aln_from_device_rows(pfa_ctx* ctx, const uint8_t* d_text, int64_t n, int64_t L, int64_t ld,
                             int64_t col_begin, int64_t col_end, pfa_aln** out);
/* deterministic synthetic alignment (pure ACGT), generated directly in packed form on the device;
 * columns [col_begin, col_end) of the n x L alignment defined by (seed, p_seg_ppm, tri_ppm).
 * The same generator exists on the host in polyfasta_b200/synth.py (numpy). */
int pfa_aln_synthetic(pfa_ctx* ctx, int64_t n, int64_t L, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm,
                      int64_t col_begin, int64_t col_end, pfa_aln** out);
/* the same synthetic alignment as upper-case text d_text[row*ld + (col-col_begin)] in DEVICE memory (benchmark input
 * for the end-to-end leg: copied to pinned host memory, then uploaded like any other alignment) */
/* benchmarks / tests: turn gap_ppm cells per million of a resident alignment into '-' (deterministic in seed, site, row;
 * polyfasta_b200.synth.poke_gaps is the numpy twin).  gap_ppm <= 31250. */
int pfa_aln_poke_gaps(pfa_aln* a, uint64_t seed, uint32_t gap_ppm);
int pfa_synth_text_device(pfa_ctx* ctx, uint8_t* d_text, int64_t ld, int64_t n, uint64_t seed, uint32_t p_seg_ppm,
                          uint32_t tri_ppm, int64_t col_begin, int64_t col_end);
int pfa_aln_free(pfa_aln* a);
int64_t pfa_aln_nseq(const pfa_aln* a);
int64_t pfa_aln_nsites(const pfa_aln* a);        /* sites in this shard */
int64_t pfa_aln_total_sites(const pfa_aln* a);   /* sites of the whole alignment the shard belongs to */
int64_t pfa_aln_num_escapes(const pfa_aln* a);   /* entries in the exception list */
int64_t pfa_aln_packed_bytes(const pfa_aln* a);  /* bytes of the three planes */
int pfa_aln_has_invalid(const pfa_aln* a);       /* any non-ACGT symbol in the shard */
/* where the planes live: 0 = the device's stream-ordered pool, 1 = a virtual-memory range (cuMemCreate), 2 = the same, in
 * compressible memory.  PFA_PLANE_ALLOC = pool | vmm | compressible (default) chooses for planes of at least
 * PFA_PLANE_ALLOC_MIN_BYTES (default 64 MB); a device that does not grant compression gets 1 or 0 */
int pfa_aln_plane_alloc(const pfa_aln* a);
/* benchmarking: force the scans to read the validity plane even though the shard is pure ACGT (flag != 0) */
int pfa_aln_force_validity(pfa_aln* a, int flag);
/* measurement aid (bench.py): time `reps` passes of a kernel that only READS the first `planes` planes of this shard with the
 * scans' streaming 128-bit loads: the read-only ceiling of this GPU for exactly these bytes */
int pfa_aln_read_probe(pfa_aln* a, int planes, int reps, double* ms_per_pass);
/* debugging / tests: copy plane p (0=b0,1=b1,2=v) to the host, nsites*Wq*16 bytes */
int pfa_aln_copy_plane(pfa_aln* a, int plane, void* dst, size_t cap);

/* ---- populations: replaces the header-substring split (PolyFastA.py:123-134) ------------------------ */
/* k row bit-masks, each pfa_aln_mask_words(a) uint32 long (bit r%32 of word r/32 = row r; the words of a site record,
 * 4*Wq).  Substring matching stays in Python; an empty population never reaches the library. k = 0 restores "all rows". */
int64_t pfa_aln_mask_words(const pfa_aln* a);
int pfa_aln_set_pops(pfa_aln* a, const uint32_t* masks, int k);
int pfa_aln_num_pops(const pfa_aln* a);
int64_t pfa_aln_pop_size(const pfa_aln* a, int pop);

/* ---- K2 site scan: replaces getvarsites + the sums of nucleotide_diversity / wattersons_theta / getsfs
 *      (PolyFastA.py:252-261, 274-282, 485-497) -------------------------------------------------------- */
/* Layout of the int64 result vector: for pop q at offset pfa_site_offset(a,q): [S, H, sfs[0..n_q/2)].
 * H = sum over columns of n^2 - sum_a c_a^2 (so pi_tot = H/(n(n-1))). */
int64_t pfa_site_len(const pfa_aln* a);
int64_t pfa_site_offset(const pfa_aln* a, int pop);
/* asynchronous, result stays in device memory (d_out: int64[pfa_site_len]); the caller may all-reduce
 * it (NCCL, sum) across column shards and then read it.  d_isvar (optional, may be NULL): uint8
 * [k][nsites], 1 where the column is variable in that population. */
int pfa_site_stats_device(pfa_aln* a, int64_t* d_out, uint8_t* d_isvar);
/* synchronous convenience: same, copied to host memory */
int pfa_site_stats(pfa_aln* a, int64_t* out, uint8_t* isvar /* host, optional */);
/* the same with the per-site H: d_hsite (optional, may be NULL) int64 [k][nsites], n^2 - sum_a c_a^2 of the column in that
 * population where it is variable, 0 elsewhere (so isvar == (hsite > 0)); zero-filled by the call.  The kernels and launch
 * plan are those of pfa_site_stats_device. */
int pfa_site_stats_hsite_device(pfa_aln* a, int64_t* d_out, uint8_t* d_isvar, int64_t* d_hsite);
int pfa_site_stats_hsite(pfa_aln* a, int64_t* out, uint8_t* isvar /* host, optional */, int64_t* hsite /* host, optional */);

/* ---- K4 codon scan: replaces getvarCDSsites + get_syn_nonsyn_cod_sites + the var-site matching
 *      (PolyFastA.py:165-170, 284-434) ------------------------------------------------------------------ */
#define PFA_CDS_NSTOPS 0
#define PFA_CDS_MISSING 1   /* already multiplied by 3 (PolyFastA.py:305) */
#define PFA_CDS_SS 2        /* S_s: number of synonymous segregating positions */
#define PFA_CDS_HS 3
#define PFA_CDS_SN 4
#define PFA_CDS_HN 5
#define PFA_CDS_SUM3 6      /* sum3_by_len[l], l = 0..64 at [6+l]: sum of 3*syncodfreq over columns with l clean codons */
#define PFA_CDS_LEN 71
/* d_out: int64[k][PFA_CDS_LEN].  first_codon_phase: (global column of this shard's first site) % 3 must be 0.
 * total_len: length of the WHOLE alignment (the trailing partial codon column belongs to the last shard).
 * d_labels (optional): uint8 [k][nsites], 0 none / 1 synonymous / 2 nonsynonymous. */
int pfa_cds_stats_device(pfa_aln* a, int64_t* d_out, uint8_t* d_labels);
int pfa_cds_stats(pfa_aln* a, int64_t* out, uint8_t* labels /* host, optional */);
/* host-side classifier tables, exposed for tests (no GPU needed):
 * labels byte for two codon indices (16*b1+4*b2+b3, A=0 C=1 G=2 T=3): bits 0-1 pos0, 2-3 pos1, 4-5 pos2 */
int pfa_codon_pair_labels(int codon_a, int codon_b);
int pfa_codon_set_labels(uint64_t sense_codon_set);
int pfa_codon_syn3(int codon);   /* 3*syncodfreq (PolyFastA.py:536-557), 0..4 */
int pfa_codon_class(int codon);  /* id of the 3-char class of PolyFastA.py:324-329, 255 for stops */

/* ---- K3 pairwise mismatches: replaces nucleotide_diversity3 (PolyFastA.py:468-480) -------------------- */
/* d_out: int64[k] sum_{i<j} d_ij per population; d_matrix (optional): int32[n][n] over all rows. */
int pfa_pairwise_device(pfa_aln* a, int64_t* d_out, int32_t* d_matrix);
int pfa_pairwise(pfa_aln* a, int64_t* out, int32_t* matrix /* host, optional */);
/* d_matrix / matrix == NULL: only the sums; the n x n matrix is then never materialised (pairs are folded inside the tiles) */

/* ---- column shards on several GPUs: the sum of the per-shard vectors, fused into the scan kernels ------------------------
 * SURVEY.md 8e: an alignment split in contiguous column ranges, one process per GPU; every statistic is a sum of exact
 * integers over the shards.  A pfa_xchg owns one "symmetric" device buffer per rank; the ranks map each other's buffer
 * (CUDA IPC over NVLink / NVSwitch peer access) and the LAST block of K2 / K4 adds the shard's vector into every
 * rank's buffer with system-scope 64-bit reductions, signals, waits for the other ranks and writes the total to d_out:
 * one launch per scan, no collective library on the data path.  All ranks must issue the same sequence of exchanges
 * (same lengths); a rank that never arrives makes the others time out (pfa_xchg_status) instead of hanging: after 4 s
 * by default, PFA_XCHG_TIMEOUT_MS or pfa_xchg_set_timeout_ms change it.  Ranks should meet on the host (a barrier after
 * their uploads) before they launch an exchange, so that the wait only has to cover launch skew.
 * Usage: create on every rank -> export -> all-gather the handles on the host -> connect -> host barrier -> scans. */
typedef struct pfa_xchg pfa_xchg;
#define PFA_XCHG_HANDLE_BYTES 64
int pfa_xchg_create(pfa_ctx* ctx, int64_t cap_words, pfa_xchg** out); /* cap_words: longest vector (int64 words) */
int pfa_xchg_destroy(pfa_xchg* x);
int64_t pfa_xchg_capacity(const pfa_xchg* x);
int pfa_xchg_export(pfa_xchg* x, void* handle /* PFA_XCHG_HANDLE_BYTES */);
int pfa_xchg_connect(pfa_xchg* x, int rank, int world, const void* handles /* world * PFA_XCHG_HANDLE_BYTES, by rank */);
/* same with the buffers already addressable (several ranks in ONE process: tests) */
void* pfa_xchg_base(const pfa_xchg* x);
int pfa_xchg_connect_ptrs(pfa_xchg* x, int rank, int world, void* const* bases);
int pfa_xchg_status(pfa_xchg* x, int* timed_out); /* synchronises the ctx stream; a reported timeout is cleared */
int pfa_xchg_set_timeout_ms(pfa_xchg* x, int64_t ms);
/* profiling: %globaltimer (ns) of the last exchange on this rank: [0] last block entered, [1] vector pushed to all ranks,
 * [2] pushes acknowledged (fence), [3] all ranks have signalled, [4] total copied to d_out, [5] block 0 of K2 started */
int pfa_xchg_stamps(pfa_xchg* x, uint64_t out[8]);
/* K2 / K4 + the sum over shards: d_out (device, this rank) receives the vector of the WHOLE alignment, laid out as
 * by pfa_site_stats_device / pfa_cds_stats_device.  d_isvar / d_labels stay per shard. */
int pfa_site_stats_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out, uint8_t* d_isvar);
int pfa_cds_stats_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out, uint8_t* d_labels);
/* K2 + K4 with ONE exchange (what --cds needs per alignment): d_out = int64[pfa_site_len(a) + PFA_CDS_LEN * k], the site vector
 * followed by the codon vectors of the whole alignment */
int pfa_site_cds_stats_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out, uint8_t* d_isvar, uint8_t* d_labels);
/* the same exchange on its own for a vector produced by another kernel (K3 pairwise sums): in place on d_buf */
int pfa_xchg_allreduce(pfa_xchg* x, int64_t* d_buf, int64_t len);
/* K3 over column shards: the per-population sums of this rank's shard, then the sum over all ranks (d_ij is additive over
 * columns); d_out (device) = int64[k] of the whole alignment on every rank */
int pfa_pairwise_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out);

/* ---- batched path for many small loci: replaces the per-file loop of --dir mode (PolyFastA.py:93-94,104) ------------- */
/* A batch is filled on the host (rows are copied into one pinned blob), then pfa_batch_run does ONE upload, three segmented
 * launches (K1b encode, K2b site scan, K5b finalise; + the escape kernel when needed) and ONE synchronisation;
 * pfa_batch_run_cds adds the segmented codon scan K4b (getvarCDSsites per file, PolyFastA.py:104,165) and its K5 entries.
 * Loci with more than 16,384 sequences (codon scan: 12,288) go through pfa_aln_*. */
typedef struct pfa_batch pfa_batch;
int64_t pfa_mask_words_for(int64_t n); /* words of one population mask for an alignment of n rows */
int pfa_batch_create(pfa_ctx* ctx, pfa_batch** out);
int pfa_batch_destroy(pfa_batch* b);
int pfa_batch_clear(pfa_batch* b);
int64_t pfa_batch_size(const pfa_batch* b);
int64_t pfa_batch_text_bytes(const pfa_batch* b);
/* masks: k * pfa_mask_words_for(n) uint32 (k = 0: one population of all rows); *index receives the locus number */
int pfa_batch_add(pfa_batch* b, const pfa_fasta* f, const uint32_t* masks, int k, int64_t* index);
int pfa_batch_add_rows(pfa_batch* b, const uint8_t* text, int64_t n, int64_t L, int64_t ld, const uint32_t* masks, int k,
                       int64_t* index);
/* a locus of the synthetic generator (the alignment pfa_aln_synthetic makes for these parameters): its text is written on the
 * device when the batch is staged -- benchmarks hold 100,000 loci resident without host text.  Add host loci first. */
int pfa_batch_add_synthetic(pfa_batch* b, int64_t n, int64_t L, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm, const uint32_t* masks,
                            int k, int64_t* index);
/* --dir in one native call: read + parse (reference semantics) + header-substring split + append of `count` files with
 * `threads` host threads, rows copied straight into the pinned blob.  status[i]: PFA_OK, PFA_ERR_NOT_FASTA, PFA_ERR_RAGGED,
 * PFA_ERR_IO, PFA_ERR_NON_ASCII or PFA_BATCH_TOO_BIG (not added: use pfa_aln_*); shape[2i], shape[2i+1] = n, L;
 * locus[i] = index in the batch or -1; hits[i*max(nkeys,1)+j] = rows whose header contains keys[j] (populations without a
 * match are not added; nkeys = 0: one population of all rows). */
#define PFA_BATCH_TOO_BIG 100
int pfa_batch_add_files(pfa_batch* b, const char* const* paths, int count, const char* const* keys, int nkeys, int threads,
                        int* status, int64_t* shape, int64_t* locus, int64_t* hits);
int pfa_batch_run(pfa_batch* b, int jc);
int pfa_batch_run_cds(pfa_batch* b, int jc);
/* the two halves of a run, for callers that scan the same resident batch more than once (benchmarks): stage = upload +
 * K1b (the planes of every locus stay in HBM), scan = K2b [+ K4b] + K5b + result copy, release frees the device side */
int pfa_batch_stage(pfa_batch* b);
int pfa_batch_scan(pfa_batch* b, int jc, int cds);
int pfa_batch_release(pfa_batch* b);
/* measurement: device time (ms, CUDA events) of K2b and of K4b in the last scan; bases and plane bytes of the batch */
int pfa_batch_kernel_ms(const pfa_batch* b, double* site_ms, double* cds_ms);
int pfa_batch_shape(const pfa_batch* b, int64_t* bases, int64_t* plane_bytes /* one plane */);
int pfa_batch_num_pops(const pfa_batch* b, int64_t locus);
/* counts = {n, S, H}; sfs (optional) n/2 bins; fin (optional) the K5 output of that (locus, population) */
int pfa_batch_result(const pfa_batch* b, int64_t locus, int pop, int64_t counts[3], int64_t* sfs, void* fin /* pfa_final_out* */);
/* codon scan of (locus, population): cds = int64[PFA_CDS_LEN] (layout PFA_CDS_*), ssites, fin2 = pfa_final_out[2] for the
 * synonymous and the nonsynonymous class (polymorphism(var_s, ssites), polymorphism(var_n, nsites), PolyFastA.py:172-173) */
int pfa_batch_result_cds(const pfa_batch* b, int64_t locus, int pop, int64_t* cds, double* ssites, void* fin2 /* pfa_final_out[2] */);
/* ingest helpers for --dir: parse many files with `threads` host threads (status[i] = PFA_OK / PFA_ERR_NOT_FASTA / ...), and
 * build the row mask of the headers containing `key` (PolyFastA.py:125); returns the number of matching rows */
/* column-sharded runs over one large file: the rank that parsed it exports WHERE its rows are (a few bytes per row; 0 bytes =
 * the file was not mapped in place, every rank parses for itself), the other ranks map the file and adopt the layout without
 * scanning it */
int64_t pfa_fasta_layout_bytes(const pfa_fasta* f);
int pfa_fasta_export_layout(const pfa_fasta* f, void* buf, int64_t cap);
int pfa_fasta_import_layout(const char* path, const void* buf, int64_t bytes, pfa_fasta** out);
int pfa_fasta_parse_files(const char* const* paths, int count, int threads, pfa_fasta** out, int* status);
int64_t pfa_fasta_match_mask(const pfa_fasta* f, const char* key, int64_t key_len, uint32_t* mask, int64_t mask_words);

/* ---- K5 finalisation in fp64 on the device: replaces polymorphism / nucleotide_diversity /
 *      wattersons_theta / Dvar / jukes_cantor_correction (PolyFastA.py:485-534) --------------------------- */
typedef struct pfa_final_in {
    int64_t n, S, H;
    double seqlen; /* int seqlen, or the float ssites / nsites in CDS mode */
    int32_t jc;
    int32_t pad;
} pfa_final_in;
typedef struct pfa_final_out {
    double pi_site, theta_site, D;
    int32_t D_is_NA; /* Dv == 0 (PolyFastA.py:508-511) */
    int32_t no_var;  /* S == 0: the row is (0,0,0,"NA") (PolyFastA.py:503-504) */
} pfa_final_out;
int pfa_finalize(pfa_ctx* ctx, const pfa_final_in* in, pfa_final_out* out, int count);
/* synonymous-site count from the integer accumulators: sum_l sum3_by_len[l] / (3 l), fp64 on the device */
int pfa_cds_ssites(pfa_ctx* ctx, const int64_t* cds_out /* [count][PFA_CDS_LEN] host */, double* ssites, int count);

/* ---- sliding windows along the alignment (beyond the reference: pi, theta and D per window) -------------------------------
 * Window i covers the global columns [i*step, min(i*step + window, L)), i = 0 .. pfa_window_count(L, window, step) - 1:
 * windows start at 0, step, 2*step, ...; the first one that reaches the end of the alignment is truncated to L and is the last;
 * step > window skips the columns between windows.  A window's (S, H) are what pfa_site_stats returns for the alignment cut to
 * the window's columns, and its pi / theta / D what K5 returns for (n, S, H, seqlen = window length, jc). */
/* number of windows (no GPU needed): min(1 + ceil(max(0, L - window) / step), ceil(L / step)), 0 for L = 0; -1 when
 * L < 0, window < 1 or step < 1 */
int64_t pfa_window_count(int64_t L, int64_t window, int64_t step);
/* asynchronous: d_counts (device) = int64 [k][nwin][2], (S, H) of THIS SHARD's columns of every window, in global window
 * coordinates (nwin from the whole alignment's length): the vectors of the column shards of an alignment add up to the whole
 * alignment's (pfa_xchg_allreduce).  Runs the site scan with the per-site H into scratch memory of the device pool. */
int pfa_site_windows_device(pfa_aln* a, int64_t window, int64_t step, int64_t* d_counts);
/* synchronous: counts (host) = int64 [k][nwin][2] as above.  window < 1 or step < 1: PFA_ERR_ARG. */
int pfa_site_windows(pfa_aln* a, int64_t window, int64_t step, int64_t* counts);

/* ---- synonymous and nonsynonymous statistics in sliding windows (beyond the reference: --cds --window) --------------------
 * Windows as above; window and step must be multiples of 3, so that no codon column straddles a window boundary, and a column
 * shard must start on a codon boundary (else PFA_ERR_ARG).  The vector of a (population, window) has PFA_CDS_WIN_LEN words:
 * words 0..70 are what pfa_cds_stats returns for the alignment cut to the window's columns (PFA_CDS_* layout; the trailing
 * partial codon column of an alignment whose length is not a multiple of 3 adds 3 to `missing` of the window that holds it),
 * word PFA_CDS_WIN_S is the S of pfa_site_stats for the same cut. */
#define PFA_CDS_WIN_LEN 72
#define PFA_CDS_WIN_S 71
/* asynchronous: d_counts (device) = int64 [k][nwin][PFA_CDS_WIN_LEN] of THIS SHARD's columns, in global window coordinates: the
 * vectors of the column shards add up to the whole alignment's.  Runs the site scan with the per-site H and the codon scan with
 * the labels, then one pass over the shard's codon columns into bins of gcd(window, step) columns and a prefix sum over the
 * bins.  Device scratch from the pool: k * nsites * 9 bytes (labels and per-site H) plus (k * 72 * nbins + 1) * 8 bytes, nbins =
 * the shard's bins of gcd(window, step) columns. */
int pfa_cds_windows_device(pfa_aln* a, int64_t window, int64_t step, int64_t* d_counts);
/* synchronous: counts (host) = int64 [k][nwin][PFA_CDS_WIN_LEN] as above */
int pfa_cds_windows(pfa_aln* a, int64_t window, int64_t step, int64_t* counts);

/* ---- divergence between populations (beyond the reference: d_xy, d_a and Hudson's F_ST) ---------------------------------
 * Pairs are the unordered pairs x < y of the populations in pfa_aln_set_pops order: p = 0 .. P-1 for (0,1), (0,2), ...,
 * (0,k-1), (1,2), ..., P = k(k-1)/2; 2 <= k <= 64 (else PFA_ERR_ARG).  Every character is an allele (A, C, G, T, '-', 'N',
 * '?' and each distinct other byte).  For a column c, Dxy_site(c) = n_x n_y - sum_a c_{x,a} c_{y,a}: the ordered pairs of
 * rows (i in x, j in y) whose characters differ at c (a row in both populations compares equal to itself).  D_xy = the sum
 * of Dxy_site over the columns, an exact int64; for the whole alignment it equals sum_{i in x, j in y} d_ij of pfa_pairwise's
 * matrix.  Windows are those of pfa_window_count above. */
typedef struct pfa_div_in {
    int64_t n_x, n_y, D; /* population sizes and D_xy over the columns */
    double seqlen;       /* number of columns (the window's length in a window) */
    double pi_x, pi_y;   /* pi_site of K5 for the two populations over the same columns: 0 when S == 0, JC-corrected with jc */
    int32_t jc;
    int32_t pad;
} pfa_div_in;
typedef struct pfa_div_out {
    double dxy, da, fst;
    int32_t fst_is_NA; /* dxy == 0 */
    int32_t undefined; /* n_x n_y == 0 or seqlen <= 0: every field is undefined */
} pfa_div_out;
/* asynchronous: d_out (device) = int64 [P], THIS SHARD's D_xy of every pair (the vectors of the column shards add up) */
int pfa_divergence_device(pfa_aln* a, int64_t* d_out);
/* asynchronous: d_counts (device) = int64 [P][nwin][2], this shard's (columns with Dxy_site > 0, D_xy) of every (pair, window),
 * in global window coordinates; the vectors of the column shards add up.  Needs P * nsites * 8 bytes of device scratch for the
 * per-site values (PFA_ERR_CUDA with a message when that allocation fails). */
int pfa_divergence_windows_device(pfa_aln* a, int64_t window, int64_t step, int64_t* d_counts);
/* fp64 on the device, in this operation order: dxy = (D / (n_x n_y)) / seqlen; with jc, x = 1 - (4/3) dxy and dxy = -0.75 log(x)
 * when x > 0 (K5's rule for pi); hw = 0.5 (pi_x + pi_y); da = dxy - hw; fst = 1 - hw / dxy (Hudson, Slatkin & Maddison 1992,
 * the estimator of Bhatia et al. 2013), fst_is_NA when dxy == 0 */
int pfa_div_finalize(pfa_ctx* ctx, const pfa_div_in* in, pfa_div_out* out, int count);
/* synchronous: counts (host) = int64 [P] D_xy of the whole alignment (of this shard for a column shard) */
int pfa_divergence(pfa_aln* a, int64_t* counts);
/* synchronous: counts (host) = int64 [P][nwin][2] as pfa_divergence_windows_device gives it.  window < 1 or step < 1:
 * PFA_ERR_ARG. */
int pfa_divergence_windows(pfa_aln* a, int64_t window, int64_t step, int64_t* counts);

/* ---- haplotype classes (beyond the reference: number of haplotypes and haplotype diversity) -------------------------------
 * Two rows are the same haplotype over a set of columns iff their (upper-cased) characters are equal at every one of them:
 * every character is an allele, as in the site scan, so 'A', '-', 'N', '?' and two different other bytes all differ;
 * equivalently, d_ij of pfa_pairwise is 0 over those columns.  rep[w][r] = the smallest row index (over all rows, whatever the
 * populations) of row r's class over THIS SHARD's columns of window w; windows are those of pfa_window_count, and window = step
 * = L gives the whole alignment as the single window.  A window that does not meet the shard is one class (rep = 0).  The rows
 * are identical over the whole alignment iff they are identical in every column shard: the classes of the alignment are the
 * common refinement of the shards' classes.  Needs nwin * n <= 2^31-1 and a shard of at most 2^31-1 sites (else PFA_ERR_ARG).
 * Builds K3's row-major planes of the marked sites and a row-ordered copy of the exception list once per alignment. */
/* asynchronous: d_rep (device) = int32 [nwin][n] */
int pfa_haplotypes_device(pfa_aln* a, int64_t window, int64_t step, int32_t* d_rep);
/* synchronous: rep (host) = int32 [nwin][n] as above */
int pfa_haplotypes(pfa_aln* a, int64_t window, int64_t step, int32_t* rep);

#ifdef __cplusplus
}
#endif
#endif
