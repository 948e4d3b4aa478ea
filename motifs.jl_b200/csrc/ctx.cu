// Context management of libmotifs_b200 (C ABI in include/motifs_b200.h).
#include "common.cuh"
#include <algorithm>

extern "C" int32_t mb200_version(void) { return 100; }

extern "C" int32_t mb200_create(mb200_ctx** out, int32_t device_id) {
    if (!out) return MB200_E_INVALID;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) return MB200_E_CUDA;     // no CPU fallback: fail loudly
    if (device_id < 0 || device_id >= ndev) return MB200_E_INVALID;
    mb200_ctx* ctx = new mb200_ctx();
    ctx->device = device_id;
    if (cudaSetDevice(device_id) != cudaSuccess) { delete ctx; return MB200_E_CUDA; }
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, device_id) != cudaSuccess) { delete ctx; return MB200_E_CUDA; }
    ctx->sm_count = p.multiProcessorCount;
    ctx->smem_optin = p.sharedMemPerBlockOptin;
    if (p.major < 10) {
        // built for sm_100a only; any other device cannot run the cubin
        delete ctx; return MB200_E_UNSUPPORTED;
    }
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return MB200_E_CUDA; }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return MB200_OK;
}

extern "C" int32_t mb200_destroy(mb200_ctx* ctx) {
    if (!ctx) return MB200_E_INVALID;
    cudaSetDevice(ctx->device);
    mb200_comm_destroy(ctx);
    if (ctx->scratch) cudaFree(ctx->scratch);
    for (int i = 0; i < BUF_N; ++i) if (ctx->bufs[i]) cudaFree(ctx->bufs[i]);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (auto& b : ctx->pool) cudaFree(b.first);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return MB200_OK;
}

extern "C" const char* mb200_last_error(const mb200_ctx* ctx) {
    return ctx ? ctx->err.c_str() : "null ctx";
}

extern "C" int32_t mb200_set_stream(mb200_ctx* ctx, void* cuda_stream) {
    if (!ctx) return MB200_E_INVALID;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return MB200_OK;
}

extern "C" int32_t mb200_last_timing(const mb200_ctx* ctx, float* out_ms8, int64_t* launches8) {
    if (!ctx) return MB200_E_INVALID;
    for (int i = 0; i < T_N; ++i) {
        if (out_ms8) out_ms8[i] = ctx->ms[i];
        if (launches8) launches8[i] = ctx->launches[i];
    }
    return MB200_OK;
}

int mb_ensure_scratch(mb200_ctx* ctx, size_t bytes) {
    if (ctx->scratch_bytes >= bytes) return MB200_OK;
    if (ctx->scratch) { cudaFree(ctx->scratch); ctx->scratch = nullptr; ctx->scratch_bytes = 0; }
    if (cudaMalloc(&ctx->scratch, bytes) != cudaSuccess) {
        cudaGetLastError();
        MB_FAIL(ctx, MB200_E_NOMEM, "cudaMalloc(%zu) for scratch failed", bytes);
    }
    ctx->scratch_bytes = bytes;
    return MB200_OK;
}

int mb_ensure_pinned(mb200_ctx* ctx, size_t bytes) {
    if (ctx->pinned_bytes >= bytes) return MB200_OK;
    if (ctx->pinned) { cudaFreeHost(ctx->pinned); ctx->pinned = nullptr; ctx->pinned_bytes = 0; }
    if (cudaMallocHost(&ctx->pinned, bytes) != cudaSuccess) {
        cudaGetLastError();
        MB_FAIL(ctx, MB200_E_NOMEM, "cudaMallocHost(%zu) failed", bytes);
    }
    ctx->pinned_bytes = bytes;
    return MB200_OK;
}

int mb_ensure_buf(mb200_ctx* ctx, int slot, size_t bytes) {
    if (ctx->buf_bytes[slot] >= bytes) return MB200_OK;
    if (ctx->bufs[slot]) { cudaFree(ctx->bufs[slot]); ctx->bufs[slot] = nullptr; ctx->buf_bytes[slot] = 0; }
    if (slot == BUF_MASK) ctx->mask_clean_bytes = 0;
    if (cudaMalloc(&ctx->bufs[slot], bytes) != cudaSuccess) {
        cudaGetLastError();
        MB_FAIL(ctx, MB200_E_NOMEM, "cudaMalloc(%zu) for buffer %d failed", bytes, slot);
    }
    ctx->buf_bytes[slot] = bytes;
    return MB200_OK;
}


// Small cache of device blocks for the sequence stores: a block is reused when it is at most 25 % (or 64 MB) larger than asked.
void* mb_pool_alloc(mb200_ctx* ctx, size_t bytes, size_t* got) {
    int best = -1;
    for (int i = 0; i < (int)ctx->pool.size(); ++i) {
        const size_t b = ctx->pool[i].second;
        if (b >= bytes && b <= bytes + std::max<size_t>(bytes / 4, (size_t)64 << 20) && (best < 0 || b < ctx->pool[best].second)) best = i;
    }
    if (best >= 0) {
        void* p = ctx->pool[best].first; *got = ctx->pool[best].second;
        ctx->pool_bytes -= *got; ctx->pool.erase(ctx->pool.begin() + best);
        return p;
    }
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        for (auto& b : ctx->pool) cudaFree(b.first);               // give the cache back and retry once
        ctx->pool.clear(); ctx->pool_bytes = 0;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    *got = bytes;
    return p;
}
void mb_pool_free(mb200_ctx* ctx, void* p, size_t bytes) {
    if (!p) return;
    if (!ctx || bytes == 0) { cudaFree(p); return; }
    ctx->pool.emplace_back(p, bytes); ctx->pool_bytes += bytes;
    while (ctx->pool.size() > 6 || ctx->pool_bytes > ((size_t)12 << 30)) {       // oldest first
        cudaFree(ctx->pool.front().first); ctx->pool_bytes -= ctx->pool.front().second; ctx->pool.erase(ctx->pool.begin());
    }
}
