// C ABI of the library: contexts, alignment upload, populations, result wrappers.  See include/polyfasta_b200.h.
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include <cuda.h>
#include <cudaTypedefs.h>

#include "pfa_common.cuh"
#include "pfa_host.h"
#include "pfa_sites.cuh"

static thread_local std::string g_error;

// ---- plane memory ----------------------------------------------------------------------------------------
// Most 128-byte lines of the planes are uniform (a monomorphic site's record is all zeros or all ones in each plane), and
// Blackwell compresses such lines between L2 and HBM in memory allocated as compressible.  Stream-ordered pools cannot ask for
// that, so large planes get their own virtual-memory range over one cuMemCreate allocation.  The driver entry points come
// through the runtime: the library links only libcudart.

struct VmmApi {
    PFN_cuDeviceGet_v2000 device_get = nullptr;
    PFN_cuDeviceGetAttribute_v2000 attribute = nullptr;
    PFN_cuMemGetAllocationGranularity_v10020 granularity = nullptr;
    PFN_cuMemCreate_v10020 create = nullptr;
    PFN_cuMemRelease_v10020 release = nullptr;
    PFN_cuMemAddressReserve_v10020 reserve = nullptr;
    PFN_cuMemAddressFree_v10020 address_free = nullptr;
    PFN_cuMemMap_v10020 map = nullptr;
    PFN_cuMemUnmap_v10020 unmap = nullptr;
    PFN_cuMemSetAccess_v10020 set_access = nullptr;
    PFN_cuMemGetAllocationPropertiesFromHandle_v10020 properties = nullptr;
    bool ok = false;
};

template <typename F>
static bool driver_entry(const char* name, F* fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        return false;
    }
    *fn = reinterpret_cast<F>(p);
    return p != nullptr;
}

static const VmmApi& vmm_api() {
    static const VmmApi api = [] {
        VmmApi v;
        v.ok = driver_entry("cuDeviceGet", &v.device_get) && driver_entry("cuDeviceGetAttribute", &v.attribute) &&
               driver_entry("cuMemGetAllocationGranularity", &v.granularity) && driver_entry("cuMemCreate", &v.create) &&
               driver_entry("cuMemRelease", &v.release) && driver_entry("cuMemAddressReserve", &v.reserve) &&
               driver_entry("cuMemAddressFree", &v.address_free) && driver_entry("cuMemMap", &v.map) &&
               driver_entry("cuMemUnmap", &v.unmap) && driver_entry("cuMemSetAccess", &v.set_access) &&
               driver_entry("cuMemGetAllocationPropertiesFromHandle", &v.properties);
        return v;
    }();
    return api;
}

static void vmm_release(pfa_vmm_range* r) {
    if (!r->ptr) return;
    const VmmApi& api = vmm_api();
    const CUdeviceptr p = reinterpret_cast<CUdeviceptr>(r->ptr);
    api.unmap(p, r->size);
    api.address_free(p, r->size);
    api.release(static_cast<CUmemGenericAllocationHandle>(r->handle));
    *r = pfa_vmm_range();
}

// a new range of at least `bytes` on the ctx's device; false (nothing held) on any failure
static bool vmm_create(pfa_ctx* ctx, size_t bytes, int want, pfa_vmm_range* out) {
    const VmmApi& api = vmm_api();
    if (!api.ok) return false;
    CUdevice dev;
    if (api.device_get(&dev, ctx->device) != CUDA_SUCCESS) return false;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = dev;
    if (want == PFA_PLANES_COMPRESSIBLE) {
        int supported = 0;
        if (api.attribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev) != CUDA_SUCCESS || !supported) return false;
        prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    }
    size_t gran = 0;
    if (api.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) return false;
    const size_t size = (size_t)pfa_round_up((int64_t)bytes, (int64_t)gran);
    CUmemGenericAllocationHandle h;
    if (api.create(&h, size, &prop, 0) != CUDA_SUCCESS) return false;
    CUdeviceptr p = 0;
    if (api.reserve(&p, size, gran, 0, 0) != CUDA_SUCCESS) {
        api.release(h);
        return false;
    }
    CUmemAccessDesc access = {};
    access.location = prop.location;
    access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    bool mapped = false;
    if (api.map(p, size, 0, h, 0) == CUDA_SUCCESS) {
        mapped = true;
        if (api.set_access(p, size, &access, 1) == CUDA_SUCCESS) {
            // what the driver granted: compression can be refused (no compression resources left, a virtualised device)
            CUmemAllocationProp got = {};
            const bool compressed = want == PFA_PLANES_COMPRESSIBLE && api.properties(&got, h) == CUDA_SUCCESS &&
                                    got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
            out->ptr = reinterpret_cast<void*>(p);
            out->size = size;
            out->handle = static_cast<unsigned long long>(h);
            out->want = want;
            out->kind = compressed ? PFA_PLANES_COMPRESSIBLE : PFA_PLANES_VMM;
            return true;
        }
    }
    if (mapped) api.unmap(p, size);
    api.address_free(p, size);
    api.release(h);
    return false;
}

// PFA_PLANE_ALLOC = pool | vmm | compressible (default) for planes of at least PFA_PLANE_ALLOC_MIN_BYTES (default 64 MB); both
// are read at every allocation so that one process can compare the kinds
static int plane_alloc_wanted(size_t bytes) {
    int want = PFA_PLANES_COMPRESSIBLE;
    if (const char* e = getenv("PFA_PLANE_ALLOC")) {
        if (!strcmp(e, "pool")) want = PFA_PLANES_POOL;
        else if (!strcmp(e, "vmm")) want = PFA_PLANES_VMM;
    }
    size_t min_bytes = (size_t)64 << 20;
    if (const char* e = getenv("PFA_PLANE_ALLOC_MIN_BYTES")) min_bytes = (size_t)strtoull(e, nullptr, 10);
    return bytes >= min_bytes ? want : PFA_PLANES_POOL;
}

// the planes of `a`: the ctx's cached range when it fits, a new range, or (no VMM wanted, or any failure) the pool
static cudaError_t plane_alloc(pfa_ctx* ctx, pfa_aln* a, size_t bytes) {
    const int want = plane_alloc_wanted(bytes);
    if (want != PFA_PLANES_POOL) {
        pfa_vmm_range& c = ctx->plane_cache;
        if (c.ptr && (c.want != want || c.size < bytes)) {
            // kernels of earlier alignments may still read the cached range
            const cudaError_t e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) return e;
            vmm_release(&c);
        }
        if (c.ptr || vmm_create(ctx, bytes, want, &c)) {
            a->plane_vmm = c;
            c = pfa_vmm_range();
            a->planes = static_cast<uint4*>(a->plane_vmm.ptr);
            a->plane_alloc = a->plane_vmm.kind;
            return cudaSuccess;
        }
    }
    a->plane_alloc = PFA_PLANES_POOL;
    return pfa_dmalloc(ctx, &a->planes, bytes);
}

// the planes of a freed alignment go back to the ctx's cache; of two ranges the larger one stays
static void plane_free(pfa_ctx* ctx, pfa_aln* a) {
    if (a->plane_alloc == PFA_PLANES_POOL) {
        pfa_dfree(ctx, a->planes);
        return;
    }
    pfa_vmm_range& c = ctx->plane_cache;
    if (c.ptr) {
        cudaStreamSynchronize(ctx->stream);
        if (c.size >= a->plane_vmm.size) {
            vmm_release(&a->plane_vmm);
            return;
        }
        vmm_release(&c);
    }
    c = a->plane_vmm;
    a->plane_vmm = pfa_vmm_range();
}

void pfa_set_global_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
}

int pfa_fail(pfa_ctx* ctx, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    g_error = buf;
    return code;
}


void pfa_note_kernel(pfa_ctx* ctx, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    ctx->last_kernel = buf;
}

// run a *_device entry point into temporary device buffers and copy the results to the host
template <typename F>
static int run_to_host(pfa_aln* a, size_t out_bytes, void* out, size_t aux_bytes, void* aux, F launch) {
    pfa_ctx* ctx = a->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    void *d_out = nullptr, *d_aux = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &d_out, std::max<size_t>(out_bytes, 8)));
    if (aux) {
        cudaError_t e = pfa_dmalloc(ctx, &d_aux, std::max<size_t>(aux_bytes, 8));
        if (e != cudaSuccess) {
            pfa_dfree(ctx, d_out);
            return pfa_fail(ctx, PFA_ERR_CUDA, "cudaMalloc failed: %s", cudaGetErrorString(e));
        }
    }
    int rc = launch(d_out, d_aux);
    cudaError_t e = cudaSuccess;
    if (!rc) {
        e = cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess && aux && aux_bytes) e = cudaMemcpyAsync(aux, d_aux, aux_bytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    pfa_dfree(ctx, d_out);
    pfa_dfree(ctx, d_aux);
    if (rc) return rc;
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "result copy failed: %s", cudaGetErrorString(e));
    return PFA_OK;
}

extern "C" {

int pfa_version(void) { return 100; }
const char* pfa_global_error(void) { return g_error.c_str(); }

int pfa_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int pfa_ctx_create(int device, pfa_ctx** out) {
    if (!out) return PFA_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        pfa_set_global_error("no CUDA device available (%s); polyfasta_b200 has no CPU fallback",
                             e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return PFA_ERR_CUDA;
    }
    if (device < 0 || device >= n) {
        pfa_set_global_error("device %d out of range (0..%d)", device, n - 1);
        return PFA_ERR_ARG;
    }
    pfa_ctx* ctx = new (std::nothrow) pfa_ctx();
    if (!ctx) return PFA_ERR_NOMEM;
    ctx->device = device;
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    double t_dev = 0, t_streams = 0;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        pfa_set_global_error("cannot initialise device %d: %s", device, cudaGetErrorString(e));
        delete ctx;
        return PFA_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    t_dev = since();
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 3; ++i) {
        cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ctx->ev_encoded[i], cudaEventDisableTiming | cudaEventBlockingSync);  // the ingest lanes sleep on these
    }
    cudaEventCreateWithFlags(&ctx->ev_ready, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&ctx->enc_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->pack_stream, cudaStreamNonBlocking);
    for (auto& ev : ctx->ev_slot) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming | cudaEventBlockingSync);
    for (auto& ev : ctx->ev_slot_copied) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto& ev : ctx->ev_join) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    cudaGetLastError();
    t_streams = since();
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) ctx->sm_count = sms;
    if (getenv("PFA_TRACE_INIT"))
        fprintf(stderr, "[pfa ctx] set device + first stream %.1f ms, pool / streams / events %.1f ms, attributes %.1f ms\n", t_dev,
                t_streams - t_dev, since() - t_streams);
    // the codon tables go to constant memory on the first codon scan (loading that module costs a cold start ~0.1 s)
    *out = ctx;
    return PFA_OK;
}

int pfa_ctx_destroy(pfa_ctx* ctx) {
    if (!ctx) return PFA_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    vmm_release(&ctx->plane_cache);
    if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->d_work) cudaFree(ctx->d_work);
    for (int i = 0; i < 3; ++i) {
        if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
        if (ctx->ev_encoded[i]) cudaEventDestroy(ctx->ev_encoded[i]);
    }
    if (ctx->ev_ready) cudaEventDestroy(ctx->ev_ready);
    for (auto& ev : ctx->ev_slot) if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->ev_slot_copied) if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->ev_join) if (ev) cudaEventDestroy(ev);
    if (ctx->pack_pinned) cudaFreeHost(ctx->pack_pinned);
    if (ctx->raw_pinned) cudaFreeHost(ctx->raw_pinned);
    if (ctx->enc_stream) cudaStreamDestroy(ctx->enc_stream);
    if (ctx->pack_stream) cudaStreamDestroy(ctx->pack_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return PFA_OK;
}

int pfa_ctx_trim(pfa_ctx* ctx) {
    if (!ctx) return PFA_ERR_ARG;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    vmm_release(&ctx->plane_cache);
    cudaMemPool_t pool;
    PFA_CUDA(ctx, cudaDeviceGetDefaultMemPool(&pool, ctx->device));
    PFA_CUDA(ctx, cudaMemPoolTrimTo(pool, 0));
    return PFA_OK;
}

const char* pfa_last_error(const pfa_ctx* ctx) { return ctx ? ctx->err.c_str() : g_error.c_str(); }
const char* pfa_ctx_last_kernel(const pfa_ctx* ctx) { return ctx ? ctx->last_kernel.c_str() : ""; }

int pfa_ctx_sync(pfa_ctx* ctx) {
    if (!ctx) return PFA_ERR_ARG;
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFA_OK;
}

int pfa_ctx_set_stream(pfa_ctx* ctx, void* cuda_stream) {
    if (!ctx) return PFA_ERR_ARG;
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // stream-ordered allocations must not straddle two streams
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return PFA_OK;
}

int64_t pfa_ctx_launch_count(const pfa_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

// ---- upload -------------------------------------------------------------------------------------------

int pfa_aln_free(pfa_aln* a) {
    if (!a) return PFA_OK;
    pfa_ctx* ctx = a->ctx;
    cudaSetDevice(ctx->device);
    plane_free(ctx, a);
    pfa_dfree(ctx, a->vflag);
    pfa_dfree(ctx, a->exc_keys);
    pfa_dfree(ctx, a->exc_heads);
    pfa_dfree(ctx, a->d_masks);
    pfa_dfree(ctx, a->d_union);
    pfa_dfree(ctx, a->d_pop_n);
    pfa_dfree(ctx, a->rowmajor);
    pfa_dfree(ctx, a->rowmajor_sites);
    pfa_dfree(ctx, a->exc_rows);
    pfa_dfree(ctx, a->exc_row_off);
    delete a;
    return PFA_OK;
}

int pfa_aln_from_rows(pfa_ctx* ctx, const uint8_t* text, int64_t n, int64_t L, int64_t ld, int64_t col_begin, int64_t col_end,
                      pfa_aln** out) {
    return pfa_aln_from_text(ctx, text, false, n, L, ld, col_begin, col_end, out);
}

int pfa_aln_from_device_rows(pfa_ctx* ctx, const uint8_t* d_text, int64_t n, int64_t L, int64_t ld, int64_t col_begin,
                             int64_t col_end, pfa_aln** out) {
    return pfa_aln_from_text(ctx, d_text, true, n, L, ld, col_begin, col_end, out);
}

int pfa_aln_from_fasta(pfa_ctx* ctx, const pfa_fasta* f, int64_t col_begin, int64_t col_end, pfa_aln** out) {
    if (!ctx || !f || !out) return PFA_ERR_ARG;
    if (f->seqlen < 0) return pfa_fail(ctx, PFA_ERR_RAGGED, "sequences do not have the same length");
    return pfa_aln_from_text(ctx, f->data, false, f->n, f->seqlen, std::max<int64_t>(f->seqlen, 1), col_begin, col_end, out,
                             f->in_place ? f->row_off.data() : nullptr, f->wrap_w.empty() ? nullptr : f->wrap_w.data(),
                             f->wrap_gap.empty() ? nullptr : f->wrap_gap.data());
}

int pfa_aln_synthetic(pfa_ctx* ctx, int64_t n, int64_t L, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm, int64_t col_begin,
                      int64_t col_end, pfa_aln** out) {
    if (!ctx || !out) return PFA_ERR_ARG;
    *out = nullptr;
    if (n <= 0 || L <= 0 || col_begin < 0 || col_end < col_begin || col_end > L || n >= (1ll << 24))
        return pfa_fail(ctx, PFA_ERR_ARG, "bad synthetic shape");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    pfa_aln* a = nullptr;
    int rc = pfa_aln_alloc(ctx, n, L, col_begin, col_end, &a);
    if (rc) return rc;
    rc = pfa_synth_fill(a, seed, p_seg_ppm, tri_ppm);
    if (!rc) rc = pfa_aln_default_pop(a);
    if (rc) {
        pfa_aln_free(a);
        return rc;
    }
    *out = a;
    return PFA_OK;
}

int64_t pfa_aln_nseq(const pfa_aln* a) { return a ? a->n : 0; }
int64_t pfa_aln_nsites(const pfa_aln* a) { return a ? a->ns : 0; }
int64_t pfa_aln_total_sites(const pfa_aln* a) { return a ? a->L_total : 0; }
int64_t pfa_aln_num_escapes(const pfa_aln* a) { return a ? a->n_exc : 0; }
int64_t pfa_aln_packed_bytes(const pfa_aln* a) { return a ? 3 * a->ns * (int64_t)a->Wq * 16 : 0; }
int pfa_aln_has_invalid(const pfa_aln* a) { return a ? a->has_invalid : 0; }
int pfa_aln_plane_alloc(const pfa_aln* a) { return a ? a->plane_alloc : -1; }
int pfa_aln_force_validity(pfa_aln* a, int flag) {
    if (!a) return PFA_ERR_ARG;
    if (flag) a->has_invalid |= 2;
    else a->has_invalid &= 1;
    return PFA_OK;
}

int pfa_aln_copy_plane(pfa_aln* a, int plane, void* dst, size_t cap) {
    if (!a || plane < 0 || plane > 2 || !dst) return PFA_ERR_ARG;
    const size_t bytes = (size_t)a->ns * a->Wq * 16;
    if (cap < bytes) return pfa_fail(a->ctx, PFA_ERR_ARG, "plane buffer too small");
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    const uint4* src = plane == 0 ? a->b0 : plane == 1 ? a->b1 : a->v;
    PFA_CUDA(a->ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, a->ctx->stream));
    PFA_CUDA(a->ctx, cudaStreamSynchronize(a->ctx->stream));
    return PFA_OK;
}

// ---- populations ---------------------------------------------------------------------------------------

int pfa_aln_set_pops(pfa_aln* a, const uint32_t* masks, int k) {
    if (!a || k < 0 || (k > 0 && !masks)) return PFA_ERR_ARG;
    if (k == 0) return pfa_aln_default_pop(a);
    pfa_ctx* ctx = a->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t Wn = (int64_t)a->Wq * 4;
    std::vector<uint32_t> m((size_t)(k * Wn)), uni((size_t)Wn, 0u);
    a->pop_n.assign((size_t)k, 0);
    a->site_off.assign((size_t)k + 1, 0);
    std::vector<int64_t> meta((size_t)(3 * k + 1));
    int64_t sfs_total = 0;
    for (int q = 0; q < k; ++q) {
        int64_t cnt = 0;
        for (int64_t w = 0; w < Wn; ++w) {
            uint32_t x = masks[q * Wn + w];
            const int64_t lo = w * 32;
            if (lo >= a->n) x = 0;
            else if (lo + 32 > a->n) x &= (1u << (a->n - lo)) - 1u;
            m[(size_t)(q * Wn + w)] = x;
            uni[(size_t)w] |= x;
            cnt += __builtin_popcount(x);
        }
        a->pop_n[(size_t)q] = cnt;
        a->site_off[(size_t)q + 1] = a->site_off[(size_t)q] + 2 + cnt / 2;
        meta[(size_t)q] = cnt;
        meta[(size_t)(k + q)] = a->site_off[(size_t)q];
        meta[(size_t)(2 * k + q)] = sfs_total;
        sfs_total += cnt / 2;
    }
    meta[(size_t)(3 * k)] = sfs_total;
    pfa_dfree(ctx, a->d_masks);
    pfa_dfree(ctx, a->d_union);
    pfa_dfree(ctx, a->d_pop_n);
    a->d_masks = a->d_union = nullptr;
    a->d_pop_n = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &a->d_masks, sizeof(uint32_t) * (size_t)std::max<int64_t>(k * Wn, 4)));
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &a->d_union, sizeof(uint32_t) * (size_t)std::max<int64_t>(Wn, 4)));
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &a->d_pop_n, sizeof(int64_t) * meta.size()));
    if (Wn) {
        PFA_CUDA(ctx, cudaMemcpyAsync(a->d_masks, m.data(), sizeof(uint32_t) * m.size(), cudaMemcpyHostToDevice, ctx->stream));
        PFA_CUDA(ctx, cudaMemcpyAsync(a->d_union, uni.data(), sizeof(uint32_t) * uni.size(), cudaMemcpyHostToDevice, ctx->stream));
    }
    PFA_CUDA(ctx, cudaMemcpyAsync(a->d_pop_n, meta.data(), sizeof(int64_t) * meta.size(), cudaMemcpyHostToDevice, ctx->stream));
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    a->d_site_off = a->d_pop_n + k;
    a->k = k;
    return PFA_OK;
}

int pfa_aln_num_pops(const pfa_aln* a) { return a ? a->k : 0; }
int64_t pfa_aln_mask_words(const pfa_aln* a) { return a ? (int64_t)a->Wq * 4 : 0; }
int64_t pfa_aln_pop_size(const pfa_aln* a, int pop) { return (a && pop >= 0 && pop < a->k) ? a->pop_n[(size_t)pop] : -1; }
int64_t pfa_site_len(const pfa_aln* a) { return a ? a->site_off[(size_t)a->k] : 0; }
int64_t pfa_site_offset(const pfa_aln* a, int pop) { return (a && pop >= 0 && pop <= a->k) ? a->site_off[(size_t)pop] : -1; }

// ---- scans ----------------------------------------------------------------------------------------------

int pfa_site_stats_device(pfa_aln* a, int64_t* d_out, uint8_t* d_isvar) {
    if (!a || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_site_scan(a, d_out, d_isvar);
}

int pfa_site_stats(pfa_aln* a, int64_t* out, uint8_t* isvar) {
    if (!a || !out) return PFA_ERR_ARG;
    return run_to_host(a, sizeof(int64_t) * (size_t)pfa_site_len(a), out, (size_t)(a->k * a->ns), isvar,
                       [&](void* d_out, void* d_aux) { return pfa_launch_site_scan(a, (int64_t*)d_out, (uint8_t*)d_aux); });
}

int pfa_site_stats_hsite_device(pfa_aln* a, int64_t* d_out, uint8_t* d_isvar, int64_t* d_hsite) {
    if (!a || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_site_scan(a, d_out, d_isvar, nullptr, false, d_hsite);
}

int pfa_site_stats_hsite(pfa_aln* a, int64_t* out, uint8_t* isvar, int64_t* hsite) {
    if (!a || !out) return PFA_ERR_ARG;
    if (!hsite) return pfa_site_stats(a, out, isvar);
    pfa_ctx* ctx = a->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t hbytes = sizeof(int64_t) * (size_t)a->k * (size_t)a->ns;
    int64_t* d_hsite = nullptr;
    PFA_CUDA(ctx, pfa_dmalloc(ctx, &d_hsite, std::max<size_t>(hbytes, 8)));
    int rc = run_to_host(a, sizeof(int64_t) * (size_t)pfa_site_len(a), out, (size_t)(a->k * a->ns), isvar, [&](void* d_out, void* d_aux) {
        return pfa_launch_site_scan(a, (int64_t*)d_out, (uint8_t*)d_aux, nullptr, false, d_hsite);
    });
    cudaError_t e = cudaSuccess;
    if (!rc && hbytes) {
        e = cudaMemcpyAsync(hsite, d_hsite, hbytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    pfa_dfree(ctx, d_hsite);
    if (rc) return rc;
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "result copy failed: %s", cudaGetErrorString(e));
    return PFA_OK;
}

int pfa_cds_stats_device(pfa_aln* a, int64_t* d_out, uint8_t* d_labels) {
    if (!a || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_cds_scan(a, d_out, d_labels);
}

int pfa_cds_stats(pfa_aln* a, int64_t* out, uint8_t* labels) {
    if (!a || !out) return PFA_ERR_ARG;
    return run_to_host(a, sizeof(int64_t) * PFA_CDS_LEN * (size_t)a->k, out, (size_t)(a->k * a->ns), labels,
                       [&](void* d_out, void* d_aux) { return pfa_launch_cds_scan(a, (int64_t*)d_out, (uint8_t*)d_aux); });
}

int pfa_cds_windows_device(pfa_aln* a, int64_t window, int64_t step, int64_t* d_counts) {
    if (!a) return PFA_ERR_ARG;
    pfa_ctx* ctx = a->ctx;
    if (window < 1 || step < 1 || window % 3 != 0 || step % 3 != 0)
        return pfa_fail(ctx, PFA_ERR_ARG, "cds windows: window and step must be positive multiples of 3 (got %lld, %lld)", (long long)window,
                        (long long)step);
    if (a->col_begin % 3 != 0) return pfa_fail(ctx, PFA_ERR_ARG, "cds windows: the shard must start on a codon boundary");
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    if (nwin == 0) return PFA_OK;
    if (!d_counts) return pfa_fail(ctx, PFA_ERR_ARG, "cds windows: null output");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t per_site = (size_t)a->k * (size_t)a->ns;
    int64_t *d_site = nullptr, *d_cds = nullptr, *d_hsite = nullptr;
    uint8_t* d_labels = nullptr;
    cudaError_t e = pfa_dmalloc(ctx, &d_site, sizeof(int64_t) * (size_t)std::max<int64_t>(pfa_site_len(a), 1));
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_cds, sizeof(int64_t) * PFA_CDS_LEN * (size_t)a->k);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_hsite, sizeof(int64_t) * std::max<size_t>(per_site, 1));
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &d_labels, std::max<size_t>(per_site, 1));
    int rc = e == cudaSuccess ? PFA_OK : pfa_fail(ctx, PFA_ERR_CUDA, "cds windows: cudaMallocAsync failed: %s", cudaGetErrorString(e));
    if (!rc) rc = pfa_launch_site_scan(a, d_site, nullptr, nullptr, false, d_hsite);
    if (!rc) rc = pfa_launch_cds_scan(a, d_cds, d_labels);
    if (!rc) rc = pfa_launch_cds_windows(a, d_hsite, d_labels, window, step, d_counts);
    pfa_dfree(ctx, d_labels);
    pfa_dfree(ctx, d_hsite);
    pfa_dfree(ctx, d_cds);
    pfa_dfree(ctx, d_site);
    return rc;
}

int pfa_cds_windows(pfa_aln* a, int64_t window, int64_t step, int64_t* counts) {
    if (!a) return PFA_ERR_ARG;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    if (nwin <= 0) return pfa_cds_windows_device(a, window, step, nullptr);  // argument errors, or nothing to do
    if (!counts) return pfa_fail(a->ctx, PFA_ERR_ARG, "cds windows: null output");
    return run_to_host(a, sizeof(int64_t) * PFA_CDS_WIN_LEN * (size_t)(a->k * nwin), counts, 0, nullptr,
                       [&](void* d_out, void*) { return pfa_cds_windows_device(a, window, step, (int64_t*)d_out); });
}

int pfa_site_windows(pfa_aln* a, int64_t window, int64_t step, int64_t* counts) {
    if (!a) return PFA_ERR_ARG;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    if (nwin <= 0) return pfa_site_windows_device(a, window, step, nullptr);  // argument errors, or nothing to do
    if (!counts) return pfa_fail(a->ctx, PFA_ERR_ARG, "windows: null output");
    return run_to_host(a, sizeof(int64_t) * 2 * (size_t)(a->k * nwin), counts, 0, nullptr,
                       [&](void* d_out, void*) { return pfa_site_windows_device(a, window, step, (int64_t*)d_out); });
}

int pfa_divergence(pfa_aln* a, int64_t* counts) {
    if (!a || !counts) return PFA_ERR_ARG;
    const int64_t P = (int64_t)a->k * (a->k - 1) / 2;
    return run_to_host(a, sizeof(int64_t) * (size_t)P, counts, 0, nullptr,
                       [&](void* d_out, void*) { return pfa_divergence_device(a, (int64_t*)d_out); });
}

int pfa_divergence_windows(pfa_aln* a, int64_t window, int64_t step, int64_t* counts) {
    if (!a) return PFA_ERR_ARG;
    const int64_t nwin = pfa_window_count(a->L_total, window, step), P = (int64_t)a->k * (a->k - 1) / 2;
    if (nwin <= 0 || P <= 0) return pfa_divergence_windows_device(a, window, step, nullptr);  // argument errors, or nothing to do
    if (!counts) return pfa_fail(a->ctx, PFA_ERR_ARG, "divergence windows: null output");
    return run_to_host(a, sizeof(int64_t) * 2 * (size_t)(P * nwin), counts, 0, nullptr,
                       [&](void* d_out, void*) { return pfa_divergence_windows_device(a, window, step, (int64_t*)d_out); });
}

int pfa_haplotypes(pfa_aln* a, int64_t window, int64_t step, int32_t* rep) {
    if (!a) return PFA_ERR_ARG;
    const int64_t nwin = pfa_window_count(a->L_total, window, step);
    if (nwin <= 0 || a->n == 0) return pfa_haplotypes_device(a, window, step, nullptr);  // argument errors, or nothing to do
    if (!rep) return pfa_fail(a->ctx, PFA_ERR_ARG, "haplotypes: null output");
    return run_to_host(a, sizeof(int32_t) * (size_t)(nwin * a->n), rep, 0, nullptr,
                       [&](void* d_rep, void*) { return pfa_haplotypes_device(a, window, step, (int32_t*)d_rep); });
}

int pfa_site_stats_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out, uint8_t* d_isvar) {
    if (!a || !x || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_site_scan(a, d_out, d_isvar, x);
}

int pfa_cds_stats_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out, uint8_t* d_labels) {
    if (!a || !x || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_cds_scan(a, d_out, d_labels, x);
}

/* --cds over column shards with ONE exchange: the site scan leaves its vector in the exchange's buffer, the codon scan's
 * epilogue pushes both.  d_out (device) = int64[pfa_site_len + PFA_CDS_LEN * k]: the site vector, then the codon vectors. */
int pfa_site_cds_stats_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out, uint8_t* d_isvar, uint8_t* d_labels) {
    if (!a || !x || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    int rc = pfa_launch_site_scan(a, nullptr, d_isvar, x, true);
    if (rc) {
        pfa_xchg_set_carry(x, 0);
        return rc;
    }
    return pfa_launch_cds_scan(a, d_out, d_labels, x);
}

int pfa_pairwise_device(pfa_aln* a, int64_t* d_out, int32_t* d_matrix) {
    if (!a || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    return pfa_launch_pairwise(a, d_out, d_matrix);
}

/* column shards: d_ij is additive over columns, so the per-population sums of the shards of all ranks are summed by the
 * same NVLink exchange as the scans (one extra launch of one block); d_out gets the whole alignment's sums on every rank */
int pfa_pairwise_xchg(pfa_aln* a, pfa_xchg* x, int64_t* d_out) {
    if (!a || !x || !d_out) return PFA_ERR_ARG;
    PFA_CUDA(a->ctx, cudaSetDevice(a->ctx->device));
    int rc = pfa_launch_pairwise(a, d_out, nullptr);
    if (rc) return rc;
    return pfa_xchg_launch_only(x, d_out, a->k, d_out);
}

int pfa_pairwise(pfa_aln* a, int64_t* out, int32_t* matrix) {
    if (!a || !out) return PFA_ERR_ARG;
    return run_to_host(a, sizeof(int64_t) * (size_t)a->k, out, sizeof(int32_t) * (size_t)(a->n * a->n), matrix,
                       [&](void* d_out, void* d_aux) { return pfa_launch_pairwise(a, (int64_t*)d_out, (int32_t*)d_aux); });
}

}  // extern "C"

// ---- helpers ---------------------------------------------------------------------------------------------

int pfa_aln_alloc(pfa_ctx* ctx, int64_t n, int64_t L, int64_t col_begin, int64_t col_end, pfa_aln** out) {
    pfa_aln* a = new (std::nothrow) pfa_aln();
    if (!a) return pfa_fail(ctx, PFA_ERR_NOMEM, "out of host memory");
    a->ctx = ctx;
    a->n = n;
    a->L_total = L;
    a->col_begin = col_begin;
    a->ns = col_end - col_begin;
    // ceil(n/128), long site records padded to whole 32-byte sectors so that no sector is shared by two sites
    a->Wq = (int)(pfa_mask_words_for(n) / 4);
    a->plane_bytes = (size_t)pfa_round_up(std::max<int64_t>(a->ns * (int64_t)a->Wq * 16, 16), 256);
    cudaError_t e = plane_alloc(ctx, a, 3 * a->plane_bytes);
    if (e != cudaSuccess) {
        const size_t want = 3 * a->plane_bytes;
        delete a;
        return pfa_fail(ctx, PFA_ERR_CUDA, "cudaMalloc of %zu bytes for the packed alignment failed: %s", want,
                        cudaGetErrorString(e));
    }
    a->b0 = a->planes;
    a->b1 = reinterpret_cast<uint4*>(reinterpret_cast<char*>(a->planes) + a->plane_bytes);
    a->v = reinterpret_cast<uint4*>(reinterpret_cast<char*>(a->planes) + 2 * a->plane_bytes);
    a->gc = std::max(1, (a->Wq + 31) / 32);
    const size_t vf_bytes = sizeof(uint32_t) * (size_t)(a->ns + 64);
    if (e == cudaSuccess) e = pfa_dmalloc(ctx, &a->vflag, vf_bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(a->vflag, 0, vf_bytes, ctx->stream);
    // rows beyond n (padding up to a multiple of 128) must read as zero in every plane
    if (e == cudaSuccess) e = cudaMemsetAsync(a->planes, 0, 3 * a->plane_bytes, ctx->stream);
    if (e != cudaSuccess) {
        pfa_aln_free(a);
        return pfa_fail(ctx, PFA_ERR_CUDA, "cudaMemsetAsync failed: %s", cudaGetErrorString(e));
    }
    *out = a;
    return PFA_OK;
}

int pfa_aln_default_pop(pfa_aln* a) {
    const int64_t Wn = (int64_t)a->Wq * 4;
    std::vector<uint32_t> all((size_t)std::max<int64_t>(Wn, 1), 0u);
    for (int64_t r = 0; r < a->n; ++r) all[(size_t)(r >> 5)] |= 1u << (r & 31);
    return pfa_aln_set_pops(a, all.data(), 1);
}

int pfa_ctx_work(pfa_ctx* ctx, unsigned int** out) {
    if (!ctx->d_work) {
        PFA_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ctx->d_work), 256));
        PFA_CUDA(ctx, cudaMemset(ctx->d_work, 0, 256));
    }
    *out = ctx->d_work;
    return PFA_OK;
}

// number of sites of the shard whose validity flag word is not zero (counted once per alignment, one small synchronisation;
// the TMA scans size the validity area of their slots from it)
__global__ void pfa_count_flagged_kernel(const uint32_t* __restrict__ vflag, int64_t ns, unsigned long long* __restrict__ out) {
    unsigned long long c = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += (int64_t)gridDim.x * blockDim.x) c += vflag[i] != 0u;
    c = __reduce_add_sync(0xffffffffu, (unsigned)c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

int pfa_aln_flagged_sites(pfa_aln* a, int64_t* out) {
    if (a->vflag_sites < 0) {
        pfa_ctx* ctx = a->ctx;
        unsigned long long* d = nullptr;
        unsigned long long h = 0;
        PFA_CUDA(ctx, pfa_dmalloc(ctx, &d, sizeof(unsigned long long)));
        PFA_CUDA(ctx, cudaMemsetAsync(d, 0, sizeof(unsigned long long), ctx->stream));
        if (a->ns > 0 && a->vflag) {
            const unsigned blocks = (unsigned)std::min<int64_t>((a->ns + 255) / 256, (int64_t)ctx->sm_count * 8);
            pfa_count_flagged_kernel<<<blocks, 256, 0, ctx->stream>>>(a->vflag, a->ns, d);
            PFA_LAUNCH_CHECK(ctx);
        }
        PFA_CUDA(ctx, cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        pfa_dfree(ctx, d);
        a->vflag_sites = (int64_t)h;
    }
    *out = a->vflag_sites;
    return PFA_OK;
}

void pfa_fill_site_args(const pfa_aln* a, int64_t* d_out, uint8_t* d_isvar, PfaSiteArgs* args, int64_t* d_hsite) {
    memset(&args->x, 0, sizeof args->x);
    args->work = a->ctx->d_work;
    args->b0 = a->b0;
    args->b1 = a->b1;
    args->v = a->v;
    args->masks = a->d_masks;
    args->umask = a->d_union;
    args->pop_n = a->d_pop_n;
    args->out_off = a->d_pop_n + a->k;
    args->sfs_off = a->d_pop_n + 2 * a->k;
    args->out = d_out;
    args->isvar = d_isvar;
    args->hsite = d_hsite;
    args->ns = a->ns;
    args->vflag = nullptr;  // the launchers switch the sparse validity fetch on
    args->gc = a->gc;
    args->vs = 0;
    args->Wq = a->Wq;
    args->k = a->k;
    int64_t bins = 0;
    for (int q = 0; q < a->k; ++q) bins += a->pop_n[(size_t)q] / 2;
    args->sfs_bins = (int)std::min<int64_t>(bins, 1 << 30);
    args->sfs_in_smem = (16 * (int64_t)a->k + 4 * bins) <= 40 * 1024;
}
