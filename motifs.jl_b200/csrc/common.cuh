// Shared host-side plumbing of libmotifs_b200: context, error capture, event timers.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <utility>
#include "../../include/motifs_b200.h"

enum { T_PACK = 0, T_SCAN = 1, T_COUNT = 2, T_EMIT = 3, T_CSC = 4, T_H2D = 5, T_D2H = 6, T_TOTAL = 7, T_N = 8 };

// Slots of ctx->bufs.  BUF_HIST and BUF_UNITS each serve two scan modes; no single call uses both meanings of one slot.
enum {
    BUF_HIST = 0,         // scan: score histogram (mb200_scan_hist) or spacing histogram (mb200_scan_spacing)
    BUF_PLAN = 1,         // scan: tables, motif blocks, pair and emit tables, CTA ranges, counts
    BUF_MASK = 2,         // scan: hit masks or best keys of one batch (ctx->mask_clean_bytes)
    BUF_UNITS = 3,        // scan: per-unit hit counts and offsets (hit lists) or 64-bit best keys and records (best site, spacing)
    BUF_HITS = 4,         // scan: hit records of one batch
    BUF_CODES = 5,        // csc_codes: code records and counts
    BUF_SITES = 6,        // count matrices: counts, sites
    BUF_LONG_COUNT = 7,   // scan: count_long_* scratch (chromosome-scale rows)
    BUF_TC_PLAN = 8,      // tensor-core scan: B operands, slot blocks, slots
    BUF_TC_LIST = 9,      // tensor-core scan: candidate lists and counters (two sets)
    BUF_TC_UNITS = 10,    // tensor-core scan: listed units and their bitmap (two sets)
    BUF_SPACING = 11,     // spacing: anchors, thresholds, secondary lengths
    BUF_PVALUE = 12,      // p-value lookups (mb200_pvtab_lookup): keys and results of one chunk
    BUF_N = 13
};

struct mb200_ctx {
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;            // stream every kernel of this ctx is launched on
    cudaStream_t copy_stream = nullptr;       // uploads of mb200_seqs_from_ascii_async (created on first use)
    cudaStream_t aux_stream = nullptr;        // tensor-core scan: re-scoring + counting of batch i run here under the pre-filter of batch i+1
    std::string err;
    // timing of the last call
    float ms[T_N] = {0};
    int64_t launches[T_N] = {0};
    cudaEvent_t ev[2 * T_N] = {nullptr};      // start/stop per slot
    // grow-only device buffers reused across calls (bufs: one per BUF_* slot)
    void* scratch = nullptr; size_t scratch_bytes = 0;
    void* bufs[BUF_N] = {nullptr}; size_t buf_bytes[BUF_N] = {0};
    void* pinned = nullptr;  size_t pinned_bytes = 0;
    int last_scan_path = 0;                   // mb200_scan_last_path
    // freed sequence stores / staging buffers kept for the next upload (cudaMalloc + cudaFree of 0.5 GB cost 100s of ms per call)
    std::vector<std::pair<void*, size_t>> pool; size_t pool_bytes = 0;
    std::vector<int32_t> tc_cost_sig; std::vector<double> tc_cost;   // tensor-core scan: measured clocks per tile of the last block structure
    size_t mask_clean_bytes = 0;              // leading bytes of bufs[BUF_MASK] (hit masks) known to be zero (tensor-core scan path)
    // multi-GPU (csrc/comm.cu): one NCCL communicator per ctx, created by mb200_comm_init; world == 1 without one
    void* comm = nullptr; int rank = 0, world = 1;
    std::vector<mb200_hit> held_hits;         // hit list of a scan whose caller buffer was too small (mb200_scan_take_hits)
};

struct mb200_seqs {
    int64_t N = 0, Lb = 0;
    int64_t rowwords = 0;        // uint32 words per sequence = ceil(Lb/16)
    uint32_t* words = nullptr;   // device, N*rowwords (+ zeroed tail pad of PAD_WORDS)
    size_t words_bytes = 0, stage_bytes = 0;   // block sizes as handed out by mb_pool_alloc
    int device = 0;
    // asynchronous upload (mb200_seqs_from_ascii_async): rows [0, ready_end[i]) are packed once ready[i] has fired
    bool pending = false;
    std::vector<cudaEvent_t> ready; std::vector<int64_t> ready_end;
    uint8_t* stage = nullptr;    // own staging buffers + bad-symbol counter, freed by mb_seqs_finish
    cudaStream_t copy_stream = nullptr;
    // ragged store (mb200_seqs_from_ascii_ragged): row n holds hlens[n] <= Lb bases, the rest of the row is zero words.
    // A fixed-length store has ragged == false, lens == nullptr and every kernel takes its fixed-length path.
    bool ragged = false;
    int64_t* lens = nullptr;     // device, N row lengths (nullptr for a fixed store or N == 0)
    size_t lens_bytes = 0;
    std::vector<int64_t> hlens;  // host copy
};
int mb_seqs_finish(mb200_ctx* ctx, mb200_seqs* s);      // waits for a pending upload, frees its staging; MB200_E_BAD_SEQUENCE if a symbol was not A,C,G,T
static const int64_t SEQ_PAD_WORDS = 64;
int mb_seqs_alloc(mb200_ctx* ctx, int64_t N, int64_t Lb, mb200_seqs** out);   // empty store (tail pad zeroed on ctx->stream)
int mb_seqs_set_lens(mb200_ctx* ctx, mb200_seqs* s, std::vector<int64_t> hlens);   // makes s ragged: uploads the row lengths (synchronous)
static inline int64_t mb_row_len(const mb200_seqs* s, int64_t n) { return s->ragged ? s->hlens[(size_t)n] : s->Lb; }

// Effective table entry of the scan: what column j of pwm (comp = 0) or of reverse(pwm) (comp = 1: rc[b][j] = pwm[3-b][len-1-j])
// adds for base b.  greedy_search! adds pwm * onehot over all four bases, so a non-finite entry of another base turns into
// Inf * 0 = NaN (0x7E00).  pw(a, j) returns the Float16 bits of pwm entry (base a, column j).
template <class PW> static inline uint16_t mb_eff_entry(PW pw, int len, int b, int j, int comp) {
    const int jj = comp ? len - 1 - j : j;
    const uint16_t v = pw(comp ? 3 - b : b, jj);
    int others = -(int)((v & 0x7C00u) == 0x7C00u);
    for (int a = 0; a < 4; ++a) others += (pw(a, jj) & 0x7C00u) == 0x7C00u;
    return others > 0 ? (uint16_t)0x7E00u : v;
}

#define MB_FAIL(ctx, code, ...) do { char _b[512]; snprintf(_b, sizeof _b, __VA_ARGS__); \
    if (ctx) (ctx)->err = _b; return (code); } while (0)

#define MB_CUDA(ctx, expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { \
    MB_FAIL(ctx, MB200_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); } } while (0)

// Accumulating CUDA-event timer on the ctx stream.  Events are read back in mb_timers_collect().
struct MbSpan { int slot; cudaEvent_t a, b; };
struct MbTimers {
    mb200_ctx* ctx; std::vector<MbSpan> spans;
    explicit MbTimers(mb200_ctx* c) : ctx(c) {}
    int begin(int slot) {
        MbSpan s; s.slot = slot; cudaEventCreate(&s.a); cudaEventCreate(&s.b);
        cudaEventRecord(s.a, ctx->stream); spans.push_back(s); return (int)spans.size() - 1;
    }
    void end(int id) { cudaEventRecord(spans[id].b, ctx->stream); }
    int begin_on(int slot, cudaStream_t q) {
        MbSpan s; s.slot = slot; cudaEventCreate(&s.a); cudaEventCreate(&s.b);
        cudaEventRecord(s.a, q); spans.push_back(s); return (int)spans.size() - 1;
    }
    void end_on(int id, cudaStream_t q) { cudaEventRecord(spans[id].b, q); }
    void collect() {   // call after the stream was synchronised
        for (auto& s : spans) { float ms = 0; if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) ctx->ms[s.slot] += ms;
            cudaEventDestroy(s.a); cudaEventDestroy(s.b); }
        spans.clear();
    }
    ~MbTimers() { for (auto& s : spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); } }
};

int mb_ensure_scratch(mb200_ctx* ctx, size_t bytes);
int mb_ensure_pinned(mb200_ctx* ctx, size_t bytes);
int mb_ensure_buf(mb200_ctx* ctx, int slot, size_t bytes);
void* mb_pool_alloc(mb200_ctx* ctx, size_t bytes, size_t* got);   // nullptr when out of memory; *got = size of the block handed out
void mb_pool_free(mb200_ctx* ctx, void* p, size_t bytes);        // ctx may be NULL (plain cudaFree)
// collectives on device buffers, enqueued on ctx->stream; no-ops without a communicator (csrc/comm.cu)
int mb_comm_allreduce_f32(mb200_ctx* ctx, float* buf, size_t n, bool average);
int mb_comm_allreduce_u64(mb200_ctx* ctx, unsigned long long* buf, size_t n);
int mb_comm_allreduce_u32(mb200_ctx* ctx, unsigned int* buf, size_t n);
int mb_comm_broadcast_bytes(mb200_ctx* ctx, void* buf, size_t bytes, int root);
int mb_comm_allgather_bytes(mb200_ctx* ctx, const void* send, void* recv, size_t bytes_per_rank);
static inline void mb_reset_timing(mb200_ctx* ctx) { for (int i = 0; i < T_N; ++i) { ctx->ms[i] = 0; ctx->launches[i] = 0; } }
