// Sequence storage of libmotifs_b200: 2 bit/base packing on the GPU.
//
// Replaces the one-hot Float32 arrays the reference builds on the host and ships to the GPU per
// batch (loadfasta/helpers.jl:110-139 dna2dummy/data_2_dummy; inference/_h3_1_alignment.jl:74
// `cu(float_type_retrieval.(data_matrix[:,1,n:nend]))`): 16 B/bp there, 0.25 B/bp here.
// Row order A,C,G,T -> codes 0,1,2,3 follows helpers.jl:125-128.
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// ASCII -> 2 bit.  One thread per output word (16 bases).  HBM-bound: 1 B/bp read, 0.25 B/bp written.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t code_of_4(uint32_t v, uint32_t& bad) {
    // v holds 4 ASCII bytes.  (c>>1)&3 maps A->0 C->1 G->3 T->2; x^(x>>1) swaps the last two.
    uint32_t up = v & 0xDFDFDFDFu;                 // fold case
    uint32_t x = (v >> 1) & 0x03030303u;
    x ^= (x >> 1) & 0x01010101u;
    // validity: byte must be one of 0x41,0x43,0x47,0x54
    #pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t c = (up >> (8 * i)) & 0xFFu;
        bad |= !(c == 0x41u || c == 0x43u || c == 0x47u || c == 0x54u);
    }
    // gather 4 two-bit codes into the low byte
    return (x & 3u) | ((x >> 6) & 0xCu) | ((x >> 12) & 0x30u) | ((x >> 18) & 0xC0u);
}

__global__ void __launch_bounds__(256) pack_ascii_kernel(const uint8_t* __restrict__ ascii, int64_t n0, int64_t nrows,
                                                         int64_t Lb, int64_t rowwords, uint32_t* __restrict__ out,
                                                         unsigned int* __restrict__ bad_count) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nrows * rowwords) return;
    int64_t r = t / rowwords;
    int w = (int)(t - r * rowwords);
    const uint8_t* src = ascii + r * Lb + (int64_t)w * 16;
    int nb = (int)min((int64_t)16, Lb - (int64_t)w * 16);
    uint32_t word = 0, bad = 0;
    if (nb == 16 && (((uintptr_t)src) & 3u) == 0) {
        uint32_t v[4];
        if ((((uintptr_t)src) & 15u) == 0) {
            uint4 q = __ldg(reinterpret_cast<const uint4*>(src));
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
            const uint32_t* s4 = reinterpret_cast<const uint32_t*>(src);
            v[0] = __ldg(s4); v[1] = __ldg(s4 + 1); v[2] = __ldg(s4 + 2); v[3] = __ldg(s4 + 3);
        }
        #pragma unroll
        for (int i = 0; i < 4; ++i) word |= code_of_4(v[i], bad) << (8 * i);
    } else {
        for (int i = 0; i < nb; ++i) {
            uint32_t c = src[i];
            uint32_t up = c & 0xDFu;
            bad |= !(up == 0x41u || up == 0x43u || up == 0x47u || up == 0x54u);
            uint32_t x = (c >> 1) & 3u; x ^= (x >> 1);
            word |= x << (2 * i);
        }
    }
    out[(n0 + r) * rowwords + w] = word;
    if (bad) atomicAdd(bad_count, 1u);
}

// Concatenated rows of different lengths -> padded 2-bit rows.  One thread per output word; row r's bytes start at
// off[r] - off0 in the staged chunk.  Words past the row's end are written as zero (the padding every consumer relies on).
__global__ void __launch_bounds__(256) pack_ascii_ragged_kernel(const uint8_t* __restrict__ ascii, const int64_t* __restrict__ off, int64_t off0,
                                                                int64_t n0, int64_t nrows, int64_t rowwords, uint32_t* __restrict__ out,
                                                                unsigned int* __restrict__ bad_count) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nrows * rowwords) return;
    int64_t r = t / rowwords;
    int w = (int)(t - r * rowwords);
    const int64_t a = off[n0 + r], len = off[n0 + r + 1] - a;
    const uint8_t* src = ascii + (a - off0) + (int64_t)w * 16;
    const int nb = (int)max((int64_t)0, min((int64_t)16, len - (int64_t)w * 16));
    uint32_t word = 0, bad = 0;
    for (int i = 0; i < nb; ++i) {
        uint32_t c = src[i];
        uint32_t up = c & 0xDFu;
        bad |= !(up == 0x41u || up == 0x43u || up == 0x47u || up == 0x54u);
        uint32_t x = (c >> 1) & 3u; x ^= (x >> 1);
        word |= x << (2 * i);
    }
    out[(n0 + r) * rowwords + w] = word;
    if (bad) atomicAdd(bad_count, 1u);
}

// ---------------------------------------------------------------------------------------------
// one-hot Float32 (4*Lb, N) column-major -> 2 bit.  One lane per base (coalesced float4 loads),
// 16 lanes OR-reduce into one word with shuffles.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_onehot_kernel(const float4* __restrict__ onehot, int64_t n0, int64_t nrows,
                                                          int64_t Lb, int64_t rowwords, uint32_t* __restrict__ out,
                                                          unsigned int* __restrict__ bad_count) {
    // thread t -> (row r, padded base index pb in [0, rowwords*16))
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t per_row = rowwords * 16;
    int64_t r = t / per_row;
    int64_t pb = t - r * per_row;
    uint32_t code = 0, bad = 0;
    bool live = r < nrows;
    if (live && pb < Lb) {
        float4 v = __ldg(onehot + r * Lb + pb);
        bool ok = (v.x == 0.f || v.x == 1.f) && (v.y == 0.f || v.y == 1.f) && (v.z == 0.f || v.z == 1.f) &&
                  (v.w == 0.f || v.w == 1.f) && (v.x + v.y + v.z + v.w == 1.f);
        bad = !ok;
        code = (v.y != 0.f ? 1u : 0u) | (v.z != 0.f ? 2u : 0u) | (v.w != 0.f ? 3u : 0u);
    }
    uint32_t word = code << (2 * (threadIdx.x & 15));
    #pragma unroll
    for (int o = 1; o < 16; o <<= 1) word |= __shfl_xor_sync(0xffffffffu, word, o);
    if (live && (threadIdx.x & 15) == 0) out[(n0 + r) * rowwords + pb / 16] = word;
    if (bad) atomicAdd(bad_count, 1u);
}

// ---------------------------------------------------------------------------------------------
int mb_seqs_alloc(mb200_ctx* ctx, int64_t N, int64_t Lb, mb200_seqs** out) {
    if (!ctx || !out || N < 0 || Lb <= 0) MB_FAIL(ctx, MB200_E_INVALID, "seqs: bad N=%lld Lb=%lld", (long long)N, (long long)Lb);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    mb200_seqs* s = new mb200_seqs();
    s->N = N; s->Lb = Lb; s->rowwords = (Lb + 15) / 16; s->device = ctx->device;
    size_t bytes = (size_t)(N * s->rowwords + SEQ_PAD_WORDS) * 4;
    s->words = (uint32_t*)mb_pool_alloc(ctx, bytes, &s->words_bytes);
    if (!s->words) { delete s; MB_FAIL(ctx, MB200_E_NOMEM, "cudaMalloc(%zu) for sequences failed", bytes); }
    // zero the tail pad (the scan kernel reads a few words past the last sequence)
    cudaError_t e = cudaMemsetAsync(s->words + N * s->rowwords, 0, SEQ_PAD_WORDS * 4, ctx->stream);
    if (e != cudaSuccess) { mb_pool_free(ctx, s->words, s->words_bytes); delete s; MB_FAIL(ctx, MB200_E_CUDA, "memset: %s", cudaGetErrorString(e)); }
    *out = s;
    return MB200_OK;
}

static int pack_common(mb200_ctx* ctx, const void* src, bool src_on_host, bool onehot, int64_t N, int64_t Lb, mb200_seqs** out) {
    if (!src && N > 0) MB_FAIL(ctx, MB200_E_INVALID, "seqs: null input");
    mb_reset_timing(ctx);
    int rc = mb_seqs_alloc(ctx, N, Lb, out);
    if (rc) return rc;
    mb200_seqs* s = *out;
    // from here on a failure must hand the (partly packed) store back: the callers drop the handle on error
#define PC_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { mb200_seqs_free(ctx, s); *out = nullptr; \
    MB_FAIL(ctx, MB200_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); } } while (0)
    MbTimers tm(ctx);
    int t_total = tm.begin(T_TOTAL);
    const size_t bytes_per_row = onehot ? (size_t)Lb * 16 : (size_t)Lb;
    // bad-sequence counter lives at the start of scratch; staging follows
    const size_t stage_cap = (size_t)256 << 20;
    int64_t rows_per_chunk = src_on_host ? (int64_t)std::max<size_t>(1, stage_cap / bytes_per_row) : N;
    if (rows_per_chunk > N) rows_per_chunk = N;
    size_t need = 256 + (src_on_host ? (size_t)rows_per_chunk * bytes_per_row : 0);
    rc = mb_ensure_scratch(ctx, need);
    if (rc) { mb200_seqs_free(ctx, s); *out = nullptr; return rc; }
    unsigned int* d_bad = (unsigned int*)ctx->scratch;
    uint8_t* d_stage = (uint8_t*)ctx->scratch + 256;
    PC_CUDA(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
    for (int64_t n0 = 0; n0 < N; n0 += rows_per_chunk) {
        int64_t nr = std::min(rows_per_chunk, N - n0);
        const uint8_t* dsrc;
        if (src_on_host) {
            int th = tm.begin(T_H2D);
            PC_CUDA(cudaMemcpyAsync(d_stage, (const uint8_t*)src + (size_t)n0 * bytes_per_row, (size_t)nr * bytes_per_row,
                                         cudaMemcpyHostToDevice, ctx->stream));
            tm.end(th);
            dsrc = d_stage;
        } else {
            dsrc = (const uint8_t*)src + (size_t)n0 * bytes_per_row;
        }
        int tp = tm.begin(T_PACK);
        if (!onehot) {
            int64_t threads = nr * s->rowwords;
            pack_ascii_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(dsrc, n0, nr, Lb, s->rowwords, s->words, d_bad);
        } else {
            int64_t threads = nr * s->rowwords * 16;
            pack_onehot_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>((const float4*)dsrc, n0, nr, Lb, s->rowwords, s->words, d_bad);
        }
        tm.end(tp);
        ctx->launches[T_PACK] += 1;
        PC_CUDA(cudaGetLastError());
    }
    unsigned int h_bad = 0;
    PC_CUDA(cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    tm.end(t_total);
    PC_CUDA(cudaStreamSynchronize(ctx->stream));
    tm.collect();
    if (h_bad) {
        mb200_seqs_free(ctx, s); *out = nullptr;
        MB_FAIL(ctx, MB200_E_BAD_SEQUENCE, "%u words contain a symbol that is not A,C,G,T / not one-hot", h_bad);
    }
    return MB200_OK;
}
#undef PC_CUDA

extern "C" int32_t mb200_seqs_from_ascii(mb200_ctx* ctx, const uint8_t* ascii, int64_t N, int64_t Lb, mb200_seqs** out) {
    if (!ctx) return MB200_E_INVALID;
    return pack_common(ctx, ascii, true, false, N, Lb, out);
}
extern "C" int32_t mb200_seqs_from_device_ascii(mb200_ctx* ctx, const void* ascii_dev, int64_t N, int64_t Lb, mb200_seqs** out) {
    if (!ctx) return MB200_E_INVALID;
    return pack_common(ctx, ascii_dev, false, false, N, Lb, out);
}
extern "C" int32_t mb200_seqs_from_onehot_f32(mb200_ctx* ctx, const float* onehot, int64_t N, int64_t Lb, mb200_seqs** out) {
    if (!ctx) return MB200_E_INVALID;
    return pack_common(ctx, onehot, true, true, N, Lb, out);
}

int mb_seqs_set_lens(mb200_ctx* ctx, mb200_seqs* s, std::vector<int64_t> hlens) {
    s->ragged = true;
    s->hlens = std::move(hlens);
    if (s->N == 0) return MB200_OK;
    const size_t bytes = (size_t)s->N * 8;
    s->lens = (int64_t*)mb_pool_alloc(ctx, bytes, &s->lens_bytes);
    if (!s->lens) MB_FAIL(ctx, MB200_E_NOMEM, "cudaMalloc(%zu) for row lengths failed", bytes);
    MB_CUDA(ctx, cudaMemcpyAsync(s->lens, s->hlens.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
}

// Rows of different lengths: row i = ascii[offsets[i], offsets[i+1]).  Lb = the longest row (at least 1), rows padded with zero words.
// Staged like pack_common: whole rows per chunk of at most 256 MB (a longer row is a chunk of its own).
extern "C" int32_t mb200_seqs_from_ascii_ragged(mb200_ctx* ctx, const uint8_t* ascii, const int64_t* offsets, int64_t N, mb200_seqs** out) {
    if (!ctx) return MB200_E_INVALID;
    if (!out || N < 0 || !offsets) MB_FAIL(ctx, MB200_E_INVALID, "seqs_ragged: bad arguments (N=%lld)", (long long)N);
    *out = nullptr;
    std::vector<int64_t> hl((size_t)N);
    int64_t Lb = 1;
    for (int64_t i = 0; i < N; ++i) {
        hl[(size_t)i] = offsets[i + 1] - offsets[i];
        if (offsets[i] < 0 || hl[(size_t)i] < 0) MB_FAIL(ctx, MB200_E_INVALID, "seqs_ragged: offsets must be non-negative and non-decreasing (row %lld)", (long long)i);
        Lb = std::max(Lb, hl[(size_t)i]);
    }
    if (!ascii && N > 0 && offsets[N] > offsets[0]) MB_FAIL(ctx, MB200_E_INVALID, "seqs_ragged: null input");
    mb_reset_timing(ctx);
    int rc = mb_seqs_alloc(ctx, N, Lb, out);
    if (rc) return rc;
    mb200_seqs* s = *out;
    auto fail = [&](int code) { mb200_seqs_free(ctx, s); *out = nullptr; return code; };
    rc = mb_seqs_set_lens(ctx, s, hl);
    if (rc) return fail(rc);
    if (N == 0) return MB200_OK;
    MbTimers tm(ctx);
    int t_total = tm.begin(T_TOTAL);
    const size_t stage_cap = (size_t)256 << 20;
    const size_t off_bytes = ((size_t)(N + 1) * 8 + 255) & ~(size_t)255;
    size_t stage_need = 0;                                   // the largest chunk the loop below stages
    for (int64_t n0 = 0; n0 < N;) {
        int64_t n1 = n0 + 1;
        while (n1 < N && (size_t)(offsets[n1 + 1] - offsets[n0]) <= stage_cap) ++n1;
        stage_need = std::max(stage_need, (size_t)(offsets[n1] - offsets[n0]));
        n0 = n1;
    }
    rc = mb_ensure_scratch(ctx, 256 + off_bytes + stage_need);
    if (rc) return fail(rc);
    unsigned int* d_bad = (unsigned int*)ctx->scratch;
    int64_t* d_off = (int64_t*)((uint8_t*)ctx->scratch + 256);
    uint8_t* d_stage = (uint8_t*)ctx->scratch + 256 + off_bytes;
    cudaError_t e = cudaMemsetAsync(d_bad, 0, 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, offsets, (size_t)(N + 1) * 8, cudaMemcpyHostToDevice, ctx->stream);
    for (int64_t n0 = 0; n0 < N && e == cudaSuccess;) {
        int64_t n1 = n0 + 1;
        while (n1 < N && (size_t)(offsets[n1 + 1] - offsets[n0]) <= stage_cap) ++n1;
        const size_t bytes = (size_t)(offsets[n1] - offsets[n0]);
        int th = tm.begin(T_H2D);
        if (bytes) e = cudaMemcpyAsync(d_stage, ascii + offsets[n0], bytes, cudaMemcpyHostToDevice, ctx->stream);
        tm.end(th);
        int tp = tm.begin(T_PACK);
        const int64_t threads = (n1 - n0) * s->rowwords;
        pack_ascii_ragged_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(d_stage, d_off, offsets[n0], n0, n1 - n0, s->rowwords, s->words, d_bad);
        tm.end(tp);
        ctx->launches[T_PACK] += 1;
        if (e == cudaSuccess) e = cudaGetLastError();
        n0 = n1;
    }
    unsigned int h_bad = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream);
    tm.end(t_total);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { fail(0); MB_FAIL(ctx, MB200_E_CUDA, "seqs_ragged: %s", cudaGetErrorString(e)); }
    tm.collect();
    if (h_bad) { fail(0); MB_FAIL(ctx, MB200_E_BAD_SEQUENCE, "%u words contain a symbol that is not A,C,G,T", h_bad); }
    return MB200_OK;
}

extern "C" int32_t mb200_seqs_lengths(const mb200_seqs* s, int64_t* out) {
    if (!s || (!out && s->N > 0)) return MB200_E_INVALID;
    for (int64_t n = 0; n < s->N; ++n) out[n] = mb_row_len(s, n);
    return MB200_OK;
}

// Asynchronous upload: H2D copies (64 MB chunks, two staging buffers) and pack kernels are queued on the ctx's copy stream and the
// call returns; an event per chunk tells mb200_scan which sequences are ready, so the scan of the first batch starts while later
// chunks are still crossing PCIe.  The host buffer must stay valid (and should be pinned) until the first scan of these sequences
// or mb200_seqs_wait has returned.
extern "C" int32_t mb200_seqs_from_ascii_async(mb200_ctx* ctx, const uint8_t* ascii, int64_t N, int64_t Lb, mb200_seqs** out) {
    if (!ctx) return MB200_E_INVALID;
    if (!ascii && N > 0) MB_FAIL(ctx, MB200_E_INVALID, "seqs: null input");
    int rc = mb_seqs_alloc(ctx, N, Lb, out);
    if (rc) return rc;
    mb200_seqs* s = *out;
    if (N == 0) return MB200_OK;
    if (!ctx->copy_stream && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { mb200_seqs_free(ctx, s); *out = nullptr; MB_FAIL(ctx, MB200_E_CUDA, "seqs: cannot create the copy stream"); }
    const size_t chunk_bytes = (size_t)64 << 20;
    const int64_t rows_per_chunk = std::min<int64_t>(N, (int64_t)std::max<size_t>(1, chunk_bytes / (size_t)Lb));
    const size_t buf = ((size_t)rows_per_chunk * (size_t)Lb + 255) & ~(size_t)255;
    s->stage = (uint8_t*)mb_pool_alloc(ctx, 256 + 2 * buf, &s->stage_bytes);
    if (!s->stage) { mb200_seqs_free(ctx, s); *out = nullptr; MB_FAIL(ctx, MB200_E_NOMEM, "seqs: staging allocation failed"); }
    cudaStream_t q = ctx->copy_stream;
    s->copy_stream = q; s->pending = true;
    unsigned int* d_bad = (unsigned int*)s->stage;
    cudaError_t e = cudaMemsetAsync(d_bad, 0, 4, q);
    // the tail pad was zeroed on ctx->stream by seqs_alloc: order the copy stream after it
    cudaEvent_t ev0; cudaEventCreateWithFlags(&ev0, cudaEventDisableTiming); cudaEventRecord(ev0, ctx->stream); cudaStreamWaitEvent(q, ev0, 0); cudaEventDestroy(ev0);
    int b = 0;
    for (int64_t n0 = 0; n0 < N && e == cudaSuccess; n0 += rows_per_chunk, b ^= 1) {
        const int64_t nr = std::min(rows_per_chunk, N - n0);
        uint8_t* d_stage = s->stage + 256 + (size_t)b * buf;
        e = cudaMemcpyAsync(d_stage, ascii + (size_t)n0 * (size_t)Lb, (size_t)nr * (size_t)Lb, cudaMemcpyHostToDevice, q);
        const int64_t threads = nr * s->rowwords;
        pack_ascii_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, q>>>(d_stage, n0, nr, Lb, s->rowwords, s->words, d_bad);
        cudaEvent_t ev;
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        if (e == cudaSuccess) { e = cudaEventRecord(ev, q); s->ready.push_back(ev); s->ready_end.push_back(n0 + nr); }
        ctx->launches[T_PACK] += 1;
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { mb200_seqs_free(ctx, s); *out = nullptr; MB_FAIL(ctx, MB200_E_CUDA, "seqs: %s", cudaGetErrorString(e)); }
    return MB200_OK;
}

int mb_seqs_finish(mb200_ctx* ctx, mb200_seqs* s) {
    if (!s->pending) return MB200_OK;
    cudaError_t e = cudaStreamSynchronize(s->copy_stream);
    unsigned int h_bad = 0;
    if (e == cudaSuccess) e = cudaMemcpy(&h_bad, s->stage, 4, cudaMemcpyDeviceToHost);
    for (auto ev : s->ready) cudaEventDestroy(ev);
    s->ready.clear(); s->ready_end.clear();
    mb_pool_free(ctx, s->stage, s->stage_bytes); s->stage = nullptr; s->pending = false;
    if (e != cudaSuccess) MB_FAIL(ctx, MB200_E_CUDA, "seqs: upload failed: %s", cudaGetErrorString(e));
    if (h_bad) MB_FAIL(ctx, MB200_E_BAD_SEQUENCE, "%u words contain a symbol that is not A,C,G,T", h_bad);
    return MB200_OK;
}

extern "C" int32_t mb200_seqs_wait(mb200_ctx* ctx, mb200_seqs* s) {
    if (!ctx || !s) return MB200_E_INVALID;
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    return mb_seqs_finish(ctx, s);
}

extern "C" int32_t mb200_seqs_free(mb200_ctx* ctx, mb200_seqs* s) {
    if (!s) return MB200_E_INVALID;
    if (ctx) cudaSetDevice(ctx->device);
    if (s->pending) { cudaStreamSynchronize(s->copy_stream); for (auto ev : s->ready) cudaEventDestroy(ev); mb_pool_free(ctx, s->stage, s->stage_bytes); s->pending = false; }
    if (s->words) mb_pool_free(ctx, s->words, s->words_bytes);
    if (s->lens) mb_pool_free(ctx, s->lens, s->lens_bytes);
    delete s;
    return MB200_OK;
}

extern "C" int32_t mb200_seqs_shape(const mb200_seqs* s, int64_t* N, int64_t* Lb, int64_t* words_per_seq) {
    if (!s) return MB200_E_INVALID;
    if (N) *N = s->N;
    if (Lb) *Lb = s->Lb;
    if (words_per_seq) *words_per_seq = s->rowwords;
    return MB200_OK;
}

extern "C" int32_t mb200_seqs_download(mb200_ctx* ctx, const mb200_seqs* s, uint32_t* out_words, int64_t n_words) {
    if (!ctx || !s || !out_words) return MB200_E_INVALID;
    if (s->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(s)); if (rc) return rc; }
    if (n_words != s->N * s->rowwords) MB_FAIL(ctx, MB200_E_INVALID, "download: expected %lld words", (long long)(s->N * s->rowwords));
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    MB_CUDA(ctx, cudaMemcpyAsync(out_words, s->words, (size_t)n_words * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
}
