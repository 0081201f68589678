// Host side of the in-kernel NVLink exchange (pfa_xchg.cuh): symmetric buffers, CUDA IPC export / import, and the
// scan entry points that fuse K2 / K4 with the sum over column shards.  One process per GPU; the handles travel
// between the processes through whatever the host uses for plumbing (torch.distributed all_gather in
// polyfasta_b200/parallel.py).
#include <cstdlib>
#include <cstring>
#include <new>

#include "pfa_common.cuh"
#include "pfa_xchg.cuh"

struct pfa_xchg {
    pfa_ctx* ctx = nullptr;
    int64_t cap = 0;
    size_t bytes = 0;
    char* base = nullptr;                 // own symmetric buffer (cudaMalloc)
    unsigned long long* partial = nullptr;  // [cap]
    unsigned int* ticket = nullptr;       // ticket, status
    int rank = 0, world = 0;
    unsigned int epoch = 0;  // exchanges LAUNCHED so far (pfa_xchg_commit): a call that fails before its launch leaves it alone
    int high_water = 0;
    unsigned long long timeout_ns = PFA_XCHG_TIMEOUT_NS;
    bool distinct_devices = false;
    int64_t carry = 0;  // words a scan has already left in `partial` for the NEXT exchange to push along (pfa_site_cds_stats_xchg)  // connected over CUDA IPC: every rank has a GPU of its own (the wide epilogue needs that)
    char* peer[PFA_XCHG_MAX_RANKS] = {};
    bool opened[PFA_XCHG_MAX_RANKS] = {};  // mapped with cudaIpcOpenMemHandle (to be closed)
};

__global__ void __launch_bounds__(256) pfa_xchg_only_kernel(const PfaXchgDev x, const int64_t* __restrict__ src) {
    // the vector of a rank that had nothing to scan (or of a kernel without a fused epilogue, e.g. K3): add it into
    // the partial buffer, then run the same exchange as the scan kernels
    if (src)
        for (int i = threadIdx.x; i < x.len; i += blockDim.x) x.partial[i] = (unsigned long long)src[i];
    pfa_xchg_epilogue(x);
}

// coresident: the kernel this exchange is compiled into is launched with at most one block per SM slot, so that all of its blocks
// are resident together and may wait for one another (the TMA scans: one CTA per SM)
int pfa_xchg_fill(pfa_xchg* x, int64_t len, int64_t* d_out, PfaXchgDev* dev, bool coresident) {
    pfa_ctx* ctx = x->ctx;
    if (x->world <= 0) return pfa_fail(ctx, PFA_ERR_ARG, "exchange is not connected");
    if (len < 0 || len > x->cap) return pfa_fail(ctx, PFA_ERR_ARG, "exchange of %lld words exceeds the capacity %lld", (long long)len, (long long)x->cap);
    if ((int)len > x->high_water) x->high_water = (int)len;
    dev->world = x->world;
    dev->rank = x->rank;
    dev->epoch = x->epoch;
    dev->len = (int)len;
    dev->zero_len = x->high_water;
    dev->wide = coresident && x->distinct_devices && x->world > 1;
    dev->cap = x->cap;
    dev->timeout_ns = x->timeout_ns;
    dev->partial = x->partial;
    dev->ticket = x->ticket;
    dev->status = x->ticket + 1;
    dev->stamps = reinterpret_cast<unsigned long long*>(x->ticket + 16);
    dev->out = d_out;
    for (int p = 0; p < PFA_XCHG_MAX_RANKS; ++p) dev->base[p] = p < x->world ? x->peer[p] : nullptr;
    return PFA_OK;
}

unsigned long long* pfa_xchg_partial(pfa_xchg* x) { return x->partial; }
int64_t pfa_xchg_carry(const pfa_xchg* x) { return x->carry; }
void pfa_xchg_set_carry(pfa_xchg* x, int64_t words) { x->carry = words; }
int64_t pfa_xchg_cap(const pfa_xchg* x) { return x->cap; }

// the kernel that carries exchange number x->epoch is in the stream: the next launch uses the other slot.  Called only
// after a successful launch, so that an argument or launch error leaves this rank in step with its peers.
void pfa_xchg_commit(pfa_xchg* x) { x->epoch++; }

int pfa_xchg_launch_only(pfa_xchg* x, const int64_t* d_src, int64_t len, int64_t* d_out) {
    PfaXchgDev dev;
    int rc = pfa_xchg_fill(x, len, d_out, &dev, false);
    if (rc) return rc;
    pfa_xchg_only_kernel<<<1, 256, 0, x->ctx->stream>>>(dev, d_src);
    PFA_LAUNCH_CHECK(x->ctx);
    pfa_xchg_commit(x);
    return PFA_OK;
}

extern "C" {

int pfa_xchg_create(pfa_ctx* ctx, int64_t cap_words, pfa_xchg** out) {
    if (!ctx || !out || cap_words <= 0 || cap_words > (1ll << 28)) return PFA_ERR_ARG;
    *out = nullptr;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    pfa_xchg* x = new (std::nothrow) pfa_xchg();
    if (!x) return pfa_fail(ctx, PFA_ERR_NOMEM, "out of host memory");
    x->ctx = ctx;
    if (const char* e = getenv("PFA_XCHG_TIMEOUT_MS")) {
        const long long ms = atoll(e);
        if (ms > 0) x->timeout_ns = (unsigned long long)ms * 1000000ull;
    }
    x->cap = pfa_round_up(cap_words, 32);
    x->bytes = PFA_XCHG_FLAG_BYTES + sizeof(int64_t) * 2 * (size_t)x->cap;
    // plain cudaMalloc: pool (cudaMallocAsync) memory cannot be exported with cudaIpcGetMemHandle
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&x->base), x->bytes);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&x->partial), sizeof(int64_t) * (size_t)x->cap);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&x->ticket), 256);
    if (e == cudaSuccess) e = cudaMemset(x->base, 0, x->bytes);
    if (e == cudaSuccess) e = cudaMemset(x->partial, 0, sizeof(int64_t) * (size_t)x->cap);
    if (e == cudaSuccess) e = cudaMemset(x->ticket, 0, 256);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(x->base);
        cudaFree(x->partial);
        cudaFree(x->ticket);
        delete x;
        return pfa_fail(ctx, PFA_ERR_CUDA, "exchange buffers: %s", cudaGetErrorString(e));
    }
    *out = x;
    return PFA_OK;
}

int pfa_xchg_destroy(pfa_xchg* x) {
    if (!x) return PFA_OK;
    cudaSetDevice(x->ctx->device);
    cudaStreamSynchronize(x->ctx->stream);
    for (int p = 0; p < PFA_XCHG_MAX_RANKS; ++p)
        if (x->opened[p] && x->peer[p]) cudaIpcCloseMemHandle(x->peer[p]);
    cudaFree(x->base);
    cudaFree(x->partial);
    cudaFree(x->ticket);
    cudaGetLastError();
    delete x;
    return PFA_OK;
}

int64_t pfa_xchg_capacity(const pfa_xchg* x) { return x ? x->cap : 0; }
void* pfa_xchg_base(const pfa_xchg* x) { return x ? x->base : nullptr; }

int pfa_xchg_export(pfa_xchg* x, void* handle) {
    if (!x || !handle) return PFA_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == PFA_XCHG_HANDLE_BYTES, "handle size");
    PFA_CUDA(x->ctx, cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    PFA_CUDA(x->ctx, cudaIpcGetMemHandle(&h, x->base));
    memcpy(handle, &h, sizeof h);
    return PFA_OK;
}

int pfa_xchg_connect(pfa_xchg* x, int rank, int world, const void* handles) {
    if (!x || !handles || world < 1 || world > PFA_XCHG_MAX_RANKS || rank < 0 || rank >= world) return PFA_ERR_ARG;
    pfa_ctx* ctx = x->ctx;
    if (x->world) return pfa_fail(ctx, PFA_ERR_ARG, "exchange is already connected");
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int p = 0; p < world; ++p) {
        if (p == rank) {
            x->peer[p] = x->base;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const char*>(handles) + (size_t)p * PFA_XCHG_HANDLE_BYTES, sizeof h);
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (int q = 0; q < p; ++q)
                if (x->opened[q]) {
                    cudaIpcCloseMemHandle(x->peer[q]);
                    x->opened[q] = false;
                }
            return pfa_fail(ctx, PFA_ERR_CUDA, "cudaIpcOpenMemHandle of rank %d's buffer failed: %s", p, cudaGetErrorString(e));
        }
        x->peer[p] = static_cast<char*>(ptr);
        x->opened[p] = true;
    }
    x->rank = rank;
    x->world = world;
    x->distinct_devices = true;
    return PFA_OK;
}

int pfa_xchg_connect_ptrs(pfa_xchg* x, int rank, int world, void* const* bases) {
    if (!x || !bases || world < 1 || world > PFA_XCHG_MAX_RANKS || rank < 0 || rank >= world) return PFA_ERR_ARG;
    if (x->world) return pfa_fail(x->ctx, PFA_ERR_ARG, "exchange is already connected");
    for (int p = 0; p < world; ++p) x->peer[p] = p == rank ? x->base : static_cast<char*>(bases[p]);
    x->rank = rank;
    x->world = world;
    return PFA_OK;
}

int pfa_xchg_status(pfa_xchg* x, int* timed_out) {
    if (!x || !timed_out) return PFA_ERR_ARG;
    pfa_ctx* ctx = x->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    unsigned int st = 0;
    PFA_CUDA(ctx, cudaMemcpyAsync(&st, x->ticket + 1, sizeof st, cudaMemcpyDeviceToHost, ctx->stream));
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *timed_out = (int)st;
    if (st) {  // reported once: the next exchange starts from a clean status word
        PFA_CUDA(ctx, cudaMemsetAsync(x->ticket + 1, 0, sizeof(unsigned int), ctx->stream));
        PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return PFA_OK;
}

int pfa_xchg_set_timeout_ms(pfa_xchg* x, int64_t ms) {
    if (!x || ms <= 0) return PFA_ERR_ARG;
    x->timeout_ns = (unsigned long long)ms * 1000000ull;
    return PFA_OK;
}

int pfa_xchg_stamps(pfa_xchg* x, uint64_t out[8]) {
    if (!x || !out) return PFA_ERR_ARG;
    pfa_ctx* ctx = x->ctx;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    PFA_CUDA(ctx, cudaMemcpyAsync(out, x->ticket + 16, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    PFA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFA_OK;
}

int pfa_xchg_allreduce(pfa_xchg* x, int64_t* d_buf, int64_t len) {
    if (!x || !d_buf) return PFA_ERR_ARG;
    PFA_CUDA(x->ctx, cudaSetDevice(x->ctx->device));
    return pfa_xchg_launch_only(x, d_buf, len, d_buf);
}

}  // extern "C"
