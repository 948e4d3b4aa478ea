// Exact null distribution of the scan's Float16 window score (mb200_pvtab_*): survival tables, p-value thresholds and lookups.
//
// A window's score is the sequential Float16 sum greedy_search! computes (scan.cu: s = __hadd(s, w[base][j]) from s = 0), so after
// every column it is one of the NV = 63 489 non-NaN Float16 values (-0 merged with +0).  Under a background of independent bases
// with frequencies bg, the survival function S_j(t) = P(score after j columns >= t) over those values obeys the gather recurrence
//     S_0(t) = [t <= 0],   S_{j+1}(t) = sum_b bg[b] * S_j(g_{j,b}(t)),
//     g_{j,b}(t) = the smallest value s with h16(s + w[b][j]) >= t,
// because s -> h16(s + w) is monotone non-decreasing for finite w.  Non-finite addends: w = NaN sends all mass to NaN (no term);
// w = +Inf sends every s > -Inf to +Inf (term S_j(-65504) for every t); w = -Inf sends every s < +Inf to -Inf (term S_j(-Inf) -
// S_j(+Inf) at t = -Inf only).  NaN windows are never hits and carry no mass in S.  Every term is a product of non-negative numbers
// added in a fixed order: tail probabilities keep their relative precision and two builds are bit-identical.
//
// Values are addressed by rank in value order: rank 0 = -Inf, 31 744 = +0, NV - 1 = +Inf (h16_rank / rank_h16 below).
// w is the effective table of the strand (mb_eff_entry, as the scan builds it: an entry is NaN when another entry of its column is non-finite,
// Inf * 0 in the reference's sum); the reverse strand uses reverse(pwm).  DESIGN.md §3.1c.
#include "common.cuh"
#include <algorithm>
#include <cmath>
#include <limits>
#include <numeric>

namespace {
constexpr int NV = 63489;                 // ordered non-NaN Float16 values
constexpr int ZERO_RANK = 0x7C00;         // rank of +0 (and of -0)
constexpr int PV_THREADS = 256;
// Working half of the double buffer: S_j of a batch of slots alternates between the slot's table and this scratch, so that S_m
// ends in the table.  1 GiB holds 2 113 slots; more slots run in several batches.
constexpr size_t PV_WORK_BYTES = (size_t)1 << 30;
constexpr int64_t PV_LOOKUP_CHUNK = (int64_t)1 << 22;   // lookups per device round trip

__host__ __device__ inline int h16_rank(uint32_t b) { return (b & 0x8000u) ? (int)(0xFC00u - b) : (int)(b + 0x7C00u); }
__host__ __device__ inline uint16_t rank_h16(int r) { return r < ZERO_RANK ? (uint16_t)(0xFC00 - r) : (uint16_t)(r - ZERO_RANK); }
__host__ __device__ inline bool h16_isnan(uint32_t b) { return (b & 0x7C00u) == 0x7C00u && (b & 0x03FFu) != 0; }

struct Bg4 { double b[4]; };

// S_0 of the batch's slots, written where the parity rule wants it (the table when the slot length is even).
__global__ void __launch_bounds__(PV_THREADS) k_pv_init(const int32_t* __restrict__ slot_of, const int32_t* __restrict__ len_of,
                                                        double* __restrict__ S, double* __restrict__ work) {
    const int r = blockIdx.x * PV_THREADS + threadIdx.x;
    if (r >= NV) return;
    const int i = blockIdx.y;
    double* dst = (len_of[i] & 1) ? work + (size_t)i * NV : S + (size_t)slot_of[i] * NV;
    dst[r] = r <= ZERO_RANK ? 1.0 : 0.0;
}

// Column j of the recurrence for the first gridDim.y slots of the batch (sorted by length, longest first: exactly those with
// len > j).  One thread per (slot, value rank r); per base a 16-step binary search for g over the ranks.
__global__ void __launch_bounds__(PV_THREADS) k_pv_step(const int32_t* __restrict__ slot_of, const int32_t* __restrict__ len_of,
                                                        const uint16_t* __restrict__ eff, int maxlen, int j, Bg4 bg,
                                                        double* __restrict__ S, double* __restrict__ work) {
    const int r = blockIdx.x * PV_THREADS + threadIdx.x;
    if (r >= NV) return;
    const int i = blockIdx.y, slot = slot_of[i], m = len_of[i];
    double* tab = S + (size_t)slot * NV;
    double* wk = work + (size_t)i * NV;
    const bool odd = (m - j) & 1;                            // S_j sits in the table iff m - j is even
    const double* src = odd ? wk : tab;
    double* dst = odd ? tab : wk;
    const uint16_t* w = eff + ((size_t)slot * maxlen + j) * 4;
    double acc = 0.0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const uint16_t wb = w[b];
        double term = 0.0;
        if (h16_isnan(wb)) {
            term = 0.0;
        } else if (wb == 0x7C00u) {                          // +Inf: s > -Inf -> +Inf (>= every t), -Inf -> NaN
            term = src[1];
        } else if (wb == 0xFC00u) {                          // -Inf: s < +Inf -> -Inf (only t = -Inf), +Inf -> NaN
            term = r == 0 ? fmax(0.0, src[0] - src[NV - 1]) : 0.0;
        } else {
            const __half wh = __ushort_as_half(wb);
            int lo = -1, hi = NV - 1;                        // f(hi) >= r always: h16(+Inf + w) = +Inf
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                const int f = h16_rank(__half_as_ushort(__hadd(__ushort_as_half(rank_h16(mid)), wh)));
                if (f >= r) hi = mid; else lo = mid;
            }
            term = src[hi];
        }
        acc += bg.b[b] * term;
    }
    dst[r] = acc;
}

// Per slot: s* = the smallest value with S(s*) <= p; thresh = the value just below s* (-Inf when s* = -Inf, +Inf when no value
// qualifies), so that score > thresh <=> S(score) <= p for every non-NaN score.  S is non-increasing in rank.
__global__ void k_pv_thresholds(const double* __restrict__ S, const double* __restrict__ pval, int n_slots, uint16_t* __restrict__ out) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n_slots) return;
    const double p = pval[slot >> 1];
    const double* t = S + (size_t)slot * NV;
    if (!(t[NV - 1] <= p)) { out[slot] = 0x7C00u; return; }
    int lo = -1, hi = NV - 1;                                // t[hi] <= p
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (t[mid] <= p) hi = mid; else lo = mid;
    }
    out[slot] = hi == 0 ? (uint16_t)0xFC00u : rank_h16(hi - 1);
}

__global__ void k_pv_lookup(const double* __restrict__ S, const uint16_t* __restrict__ motif, const uint8_t* __restrict__ comp,
                            const uint16_t* __restrict__ score, int64_t n, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t b = score[i];
    out[i] = h16_isnan(b) ? __longlong_as_double(0x7FF8000000000000LL)
                          : S[((size_t)motif[i] * 2 + comp[i]) * NV + h16_rank(b)];
}
}  // namespace

struct mb200_pvtab {
    int32_t K = 0;
    int device = 0;
    double* S = nullptr;          // device, 2K x NV float64, slot k*2 + comp
};

extern "C" int32_t mb200_pvtab_create(mb200_ctx* ctx, const uint16_t* pwms_f16, const int64_t* lens, int32_t K, int32_t maxlen,
                                      const double* bg, mb200_pvtab** out) {
    if (!ctx) return MB200_E_INVALID;
    if (!pwms_f16 || !lens || !bg || !out) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_create: null argument");
    *out = nullptr;
    if (K < 1 || maxlen < 1) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_create: K = %d and maxlen = %d must be >= 1", K, maxlen);
    for (int k = 0; k < K; ++k)
        if (lens[k] < 1 || lens[k] > maxlen) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_create: lens[%d] = %lld outside [1, maxlen]", k, (long long)lens[k]);
    double bsum = 0.0;
    for (int b = 0; b < 4; ++b) {
        if (!std::isfinite(bg[b]) || bg[b] < 0.0) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_create: bg[%d] = %g must be finite and >= 0", b, bg[b]);
        bsum += bg[b];
    }
    if (!(std::fabs(bsum - 1.0) <= 1e-6)) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_create: bg sums to %.9g, not 1", bsum);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));

    // effective tables [slot][col][base] of both strands (mb_eff_entry, the scan's own rule)
    const int n_slots = 2 * K;
    std::vector<uint16_t> eff((size_t)n_slots * maxlen * 4, 0);
    for (int k = 0; k < K; ++k) {
        auto pw = [&](int a, int j) { return pwms_f16[(size_t)k + (size_t)K * (a + 4 * (size_t)j)]; };
        for (int c = 0; c < 2; ++c)
            for (int j = 0; j < (int)lens[k]; ++j)
                for (int b = 0; b < 4; ++b) eff[(((size_t)k * 2 + c) * maxlen + j) * 4 + b] = mb_eff_entry(pw, (int)lens[k], b, j, c);
    }
    // slots sorted by length, longest first: column j runs the first slots of a batch
    std::vector<int32_t> order(n_slots);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lens[a >> 1] > lens[b >> 1]; });
    std::vector<int32_t> olen(n_slots);
    for (int i = 0; i < n_slots; ++i) olen[i] = (int32_t)lens[order[i] >> 1];

    const int batch = (int)std::min<size_t>((size_t)n_slots, PV_WORK_BYTES / ((size_t)NV * sizeof(double)));
    std::vector<void*> dev;
    auto free_all = [&]() { for (void* p : dev) cudaFree(p); };
    auto alloc = [&](size_t bytes) -> void* {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        dev.push_back(p);
        return p;
    };
    double* S = (double*)alloc((size_t)n_slots * NV * sizeof(double));
    double* work = (double*)alloc((size_t)batch * NV * sizeof(double));
    uint16_t* d_eff = (uint16_t*)alloc(eff.size() * sizeof(uint16_t));
    int32_t* d_slot = (int32_t*)alloc((size_t)n_slots * sizeof(int32_t));
    int32_t* d_len = (int32_t*)alloc((size_t)n_slots * sizeof(int32_t));
    if (!S || !work || !d_eff || !d_slot || !d_len) {
        free_all();
        MB_FAIL(ctx, MB200_E_NOMEM, "pvtab_create: %d slots need %.2f GB of tables plus %.2f GB of working space", n_slots,
                (double)n_slots * NV * 8 / 1e9, (double)batch * NV * 8 / 1e9);
    }
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaMemcpyAsync(d_eff, eff.data(), eff.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_slot, order.data(), order.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_len, olen.data(), olen.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st);
    Bg4 b4;
    for (int b = 0; b < 4; ++b) b4.b[b] = bg[b];
    const unsigned gx = (NV + PV_THREADS - 1) / PV_THREADS;
    for (int i0 = 0; i0 < n_slots && e == cudaSuccess; i0 += batch) {
        const int nb = std::min(batch, n_slots - i0);
        k_pv_init<<<dim3(gx, nb), PV_THREADS, 0, st>>>(d_slot + i0, d_len + i0, S, work);
        for (int j = 0, active = nb; j < olen[i0]; ++j) {
            while (active > 0 && olen[i0 + active - 1] <= j) --active;     // slots of length <= j are final
            k_pv_step<<<dim3(gx, active), PV_THREADS, 0, st>>>(d_slot + i0, d_len + i0, d_eff, maxlen, j, b4, S, work);
            }
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        free_all();
        MB_FAIL(ctx, MB200_E_CUDA, "pvtab_create: %s", cudaGetErrorString(e));
    }
    for (void* p : dev) if (p != S) cudaFree(p);
    mb200_pvtab* t = new mb200_pvtab();
    t->K = K; t->device = ctx->device; t->S = S;
    *out = t;
    return MB200_OK;
}

extern "C" int32_t mb200_pvtab_destroy(mb200_ctx* ctx, mb200_pvtab* t) {
    if (!ctx || !t) return MB200_E_INVALID;
    cudaSetDevice(t->device);
    cudaFree(t->S);
    delete t;
    return MB200_OK;
}

extern "C" int32_t mb200_pvtab_thresholds(mb200_ctx* ctx, const mb200_pvtab* t, const double* pval, uint16_t* thresh_f16) {
    if (!ctx) return MB200_E_INVALID;
    if (!t || !pval || !thresh_f16) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_thresholds: null argument");
    for (int k = 0; k < t->K; ++k)
        if (!(pval[k] >= 0.0 && pval[k] <= 1.0)) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_thresholds: pval[%d] = %g outside [0, 1]", k, pval[k]);
    MB_CUDA(ctx, cudaSetDevice(t->device));
    const int n_slots = 2 * t->K;
    double* d_p = nullptr; uint16_t* d_out = nullptr;
    MB_CUDA(ctx, cudaMalloc(&d_p, (size_t)t->K * sizeof(double)));
    if (cudaMalloc(&d_out, (size_t)n_slots * sizeof(uint16_t)) != cudaSuccess) { cudaGetLastError(); cudaFree(d_p); MB_FAIL(ctx, MB200_E_NOMEM, "pvtab_thresholds: out of memory"); }
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaMemcpyAsync(d_p, pval, (size_t)t->K * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) { k_pv_thresholds<<<(n_slots + 127) / 128, 128, 0, st>>>(t->S, d_p, n_slots, d_out); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpyAsync(thresh_f16, d_out, (size_t)n_slots * sizeof(uint16_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_p); cudaFree(d_out);
    if (e != cudaSuccess) MB_FAIL(ctx, MB200_E_CUDA, "pvtab_thresholds: %s", cudaGetErrorString(e));
    return MB200_OK;
}

extern "C" int32_t mb200_pvtab_lookup(mb200_ctx* ctx, const mb200_pvtab* t, const uint16_t* motif, const uint8_t* comp,
                                      const uint16_t* score_f16, int64_t n, double* p) {
    if (!ctx) return MB200_E_INVALID;
    if (!t || n < 0 || (n > 0 && (!motif || !comp || !score_f16 || !p))) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_lookup: bad arguments");
    for (int64_t i = 0; i < n; ++i)
        if (motif[i] >= t->K || comp[i] > 1)
            MB_FAIL(ctx, MB200_E_INVALID, "pvtab_lookup: entry %lld has motif %u, comp %u (K = %d)", (long long)i, motif[i], comp[i], t->K);
    if (n == 0) return MB200_OK;
    MB_CUDA(ctx, cudaSetDevice(t->device));
    const int64_t cap = std::min(n, PV_LOOKUP_CHUNK);
    // one grow-only block: [out f64][motif u16][score u16][comp u8], widest first so every array is aligned for any cap
    const size_t need = (size_t)cap * (8 + 2 + 2 + 1);
    if (mb_ensure_buf(ctx, BUF_PVALUE, need) != MB200_OK) return MB200_E_NOMEM;
    char* base = (char*)ctx->bufs[BUF_PVALUE];
    double* d_o = (double*)base;
    uint16_t* d_m = (uint16_t*)(base + (size_t)cap * 8);
    uint16_t* d_s = (uint16_t*)(base + (size_t)cap * 10);
    uint8_t* d_c = (uint8_t*)(base + (size_t)cap * 12);
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaSuccess;
    for (int64_t i0 = 0; i0 < n && e == cudaSuccess; i0 += cap) {
        const int64_t c = std::min(cap, n - i0);
        e = cudaMemcpyAsync(d_m, motif + i0, (size_t)c * 2, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_s, score_f16 + i0, (size_t)c * 2, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_c, comp + i0, (size_t)c, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) { k_pv_lookup<<<(unsigned)((c + 255) / 256), 256, 0, st>>>(t->S, d_m, d_c, d_s, c, d_o); e = cudaGetLastError(); }
        if (e == cudaSuccess) e = cudaMemcpyAsync(p + i0, d_o, (size_t)c * 8, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (e != cudaSuccess) MB_FAIL(ctx, MB200_E_CUDA, "pvtab_lookup: %s", cudaGetErrorString(e));
    return MB200_OK;
}

extern "C" int32_t mb200_pvtab_survival(mb200_ctx* ctx, const mb200_pvtab* t, int32_t k, int32_t comp, double* out) {
    if (!ctx) return MB200_E_INVALID;
    if (!t || !out) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_survival: null argument");
    if (k < 0 || k >= t->K || comp < 0 || comp > 1) MB_FAIL(ctx, MB200_E_INVALID, "pvtab_survival: motif %d, comp %d (K = %d)", k, comp, t->K);
    MB_CUDA(ctx, cudaSetDevice(t->device));
    std::vector<double> s(NV);
    MB_CUDA(ctx, cudaMemcpyAsync(s.data(), t->S + ((size_t)k * 2 + comp) * NV, (size_t)NV * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t b = 0; b < 65536; ++b) out[b] = h16_isnan(b) ? std::numeric_limits<double>::quiet_NaN() : s[h16_rank(b)];
    return MB200_OK;
}
