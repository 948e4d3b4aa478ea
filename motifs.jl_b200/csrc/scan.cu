// PWM scan on sm_100a: scoring, threshold, hit masks, occurrence counts, sorted hit list.
//
// Reference being replaced (paths under the reference's src/):
//   inference/_h3_1_alignment.jl:18-36   greedy_search!   — the score of motif k at start l is the
//        LEFT-TO-RIGHT Float16 running sum of pwm[k, base(l+ind-1), ind] (x is one-hot, so the four
//        products per column are one exact value and three signed zeros); kept when > 0.
//   inference/_h3_1_alignment.jl:57-99   get_pos_scores_arr / gpu_scan — fwd pass with pwm, second
//        pass with reverse(pwm) (both dims reversed = reverse complement), dense D2H + host findall.
//   inference/_s2_filter_pos_w_scores.jl:116-125 filter_position_by_best_thresh! — score .> thresh.
//   inference/_h4_overlap_ratio.jl:5-15,40-79    unique start positions, union_ranges coverage
//        (with its dropped-last-interval behaviour), summed over sequences.
//
// Design (see DESIGN.md):
//   * sequences are 2 bit/base in HBM; a CTA stages a tile of packed words in shared memory with
//     1-D bulk TMA (cp.async.bulk + mbarrier, double buffered); the window of one start position
//     is 4 funnel-shifted registers, so the halo is just "read 6 words instead of 2".
//   * a lane owns one (motif, strand) "slot" and scores 16 consecutive start positions of one
//     sequence at a time (8 half2 accumulators); motifs are sorted by length, 16 motifs x 2 strands
//     per warp pass.  Per PWM column the lane reads ITS 8-byte column {A,C,G,T} once (LDS.64,
//     conflict free) and a PRMT picks the two entries the position pair needs; the PRMT selectors
//     depend only on the sequence, are built once per 16-position block and shared by all lanes
//     and all motif groups.  One HADD2/HFMA2 per two cells = one correctly rounded sequential
//     Float16 add per cell, exactly the reference's rounding order.  Shared-memory traffic is
//     0.5 B per cell (a per-lane table gather would need 2 B per cell and is bound by the
//     128 B/clk/SM shared-memory port: that was v0 of this kernel, profiles/r01_scan_v0_*).
//   * threshold compare turns 16 positions x 32 slots into 32 half-words of the hit masks.
//     Counting and the sorted hit list are derived from the masks (deterministic, no atomics on
//     the hit path, no sort).
#include "common.cuh"
#include <algorithm>
#include <cstring>
#include <cstdlib>
#include <cmath>

#define GROUP_MOTIFS 16                // motifs per warp pass
#define GROUP_SLOTS 32                 // (motif, strand) slots = lanes
#define COL_BYTES 256                  // 32 slots x {A,C,G,T} halves
#define POS_BLOCK 16                   // start positions scored per lane and pass (8 half2)
#define NSEL (POS_BLOCK - 2 + MB200_MAX_MOTIF_LEN + 2)   // selector registers of one position block
#define SCAN_THREADS 512

struct __align__(16) GroupMeta {
    int32_t len;                       // columns to run (longest motif of the group)
    int32_t tab_off;                   // byte offset of the group's table inside the motif block
    int32_t npos_max;                  // max over npos[]: position blocks starting at or beyond it have nothing to score
    int32_t reserved;
    int32_t npos[GROUP_MOTIFS];        // valid start positions per motif (Lb - len_k + 1, >= 0)
    uint16_t thr[GROUP_SLOTS];         // Float16 bits per slot: max(thresh, 0), +Inf for a disabled strand / padding
};                                     // 144 bytes
static_assert(sizeof(GroupMeta) == 144, "GroupMeta must be 144 bytes");
static_assert(sizeof(mb200_best) == 8, "mb200_best must be 8 bytes");

struct MBlock {
    int64_t blob_off;                  // byte offset of this motif block's blob (tables then metas)
    int32_t blob_bytes;                // multiple of 16
    int32_t tab_bytes;                 // bytes of tables (metas follow)
    int32_t g0, ng;                    // global group range
    int32_t cost, reserved;
};

struct ScanArgs {
    const uint32_t* seqw; int64_t rowwords; int32_t W;
    int64_t chunk0, nchunks;
    uint32_t* mask; int32_t K2pad;
    const uint8_t* blob; const MBlock* mblocks; int32_t n_mblocks;
    int32_t tile_chunks; int64_t ntiles; int32_t tile_cap_words; int32_t blob_cap_bytes;
    const int64_t* cta_range;          // [gridDim.x + 1] pair ranges (pair = mblock * ntiles + tile)
    const int64_t* lens; int64_t Lb;   // ragged stores: row lengths (scan_kernel<true> only)
};

// ---------------------------------------------------------------------------------------------
// PTX helpers: shared-memory addressing, mbarrier, 1-D bulk TMA.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// issue a (possibly large) copy as <=32 KiB bulk pieces, all completing on one mbarrier
__device__ __forceinline__ void tma_load(uint32_t dst, const uint8_t* src, uint32_t bytes, uint32_t bar) {
    mbar_expect_tx(bar, bytes);
    for (uint32_t o = 0; o < bytes; o += 32768u) {
        uint32_t n = min(32768u, bytes - o);
        tma_bulk_g2s(dst + o, src + o, n, bar);
    }
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ __half2 as_h2(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }
// first packed word of position block `pb` of sequence n (16 bases per word, so a block starts on a word)
__device__ __forceinline__ int64_t block_word(int64_t gq, int32_t W16, int64_t rowwords, int64_t* n_out, int32_t* pb_out) {
    int64_t n = gq / W16;
    int32_t pb = (int32_t)(gq - n * W16);
    *n_out = n; *pb_out = pb;
    return n * rowwords + (int64_t)pb;
}

// Best-site keys (mb200_scan_best): ord() orders Float16 bit patterns like their values; only a NaN maps to 0.  A block key is
// ord(score) << 4 | (15 - u) for the best valid start u of a 16-position block (the lowest u among equal scores), 0 for none.
__device__ __forceinline__ uint32_t h16_ord(uint32_t h) { return (h & 0x8000u) ? (~h & 0xFFFFu) : (h | 0x8000u); }

// RAGGED: row n has lens[n] <= Lb bases; its start positions end Lb - lens[n] earlier than the group metas say (the "deficit").
// BEST: instead of hit-mask half-words, write one best-site key per (position block, slot) to a.mask[lq * K2pad + slot].
template <bool RAGGED, bool BEST = false>
__global__ void __launch_bounds__(SCAN_THREADS, 1) scan_kernel(const ScanArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_blob = smem;                                                        // tables + metas of one motif block
    uint32_t* s_tile0 = reinterpret_cast<uint32_t*>(smem + a.blob_cap_bytes);
    uint32_t* s_tile1 = s_tile0 + a.tile_cap_words;
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_tile1 + a.tile_cap_words);     // [0],[1] tiles, [2] blob
    int32_t* s_ticket = reinterpret_cast<int32_t*>(s_bar + 3);                     // next position block of the current tile

    const int lane = threadIdx.x & 31;
    const int64_t q_lo = a.cta_range[blockIdx.x], q_hi = a.cta_range[blockIdx.x + 1];
    if (q_lo >= q_hi) return;

    const uint32_t bar0 = smem_u32(&s_bar[0]), bar1 = smem_u32(&s_bar[1]), bar2 = smem_u32(&s_bar[2]);
    if (threadIdx.x == 0) {
        mbar_init(bar0, 1); mbar_init(bar1, 1); mbar_init(bar2, 1);
        s_ticket[0] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // tile geometry: words [lo4, hi) of the packed array feed local position blocks [t*TC, ...)
    auto tile_span = [&](int64_t tile, int64_t& lo4, uint32_t& bytes, int64_t& first, int32_t& cnt) {
        first = tile * a.tile_chunks;
        cnt = (int32_t)min((int64_t)a.tile_chunks, a.nchunks - first);
        int64_t n; int32_t c;
        int64_t lo = block_word(a.chunk0 + first, a.W, a.rowwords, &n, &c);
        int64_t hi = block_word(a.chunk0 + first + cnt - 1, a.W, a.rowwords, &n, &c) + 6;
        lo4 = lo & ~(int64_t)3;
        bytes = (uint32_t)(((hi - lo4 + 3) & ~(int64_t)3) * 4);
    };

    uint32_t phase0 = 0, phase1 = 0, phase2 = 0;
    int32_t cur_mb = -1;
    if (threadIdx.x == 0) {                                   // prefetch the first tile
        int64_t lo4, first; uint32_t bytes; int32_t cnt;
        tile_span(q_lo % a.ntiles, lo4, bytes, first, cnt);
        tma_load(smem_u32(s_tile0), reinterpret_cast<const uint8_t*>(a.seqw + lo4), bytes, bar0);
    }

    for (int64_t q = q_lo; q < q_hi; ++q) {
        const int32_t mb = (int32_t)(q / a.ntiles);
        const int64_t tile = q - (int64_t)mb * a.ntiles;
        const int buf = (int)((q - q_lo) & 1);
        const MBlock mbk = a.mblocks[mb];
        if (mb != cur_mb) {
            // every warp finished the previous pair at the __syncthreads closing the last iteration
            if (threadIdx.x == 0) tma_load(smem_u32(s_blob), a.blob + mbk.blob_off, (uint32_t)mbk.blob_bytes, bar2);
            cur_mb = mb;
            mbar_wait(bar2, phase2); phase2 ^= 1;
        }
        if (threadIdx.x == 0 && q + 1 < q_hi) {               // prefetch next tile into the other buffer
            int64_t lo4, first; uint32_t bytes; int32_t cnt;
            tile_span((q + 1) % a.ntiles, lo4, bytes, first, cnt);
            tma_load(smem_u32(buf ? s_tile0 : s_tile1), reinterpret_cast<const uint8_t*>(a.seqw + lo4), bytes, buf ? bar0 : bar1);
        }
        int64_t lo4, first; uint32_t tbytes; int32_t cnt;
        tile_span(tile, lo4, tbytes, first, cnt);
        if (buf == 0) { mbar_wait(bar0, phase0); phase0 ^= 1; } else { mbar_wait(bar1, phase1); phase1 ^= 1; }
        const uint32_t* s_tile = buf ? s_tile1 : s_tile0;
        const GroupMeta* s_meta = reinterpret_cast<const GroupMeta*>(s_blob + mbk.tab_bytes);
        const uint32_t blob_base = smem_u32(s_blob);
        const uint32_t tab_base = blob_base + lane * 8;
        for (;;) {
            int32_t i = 0;
            if (lane == 0) i = atomicAdd(s_ticket, 1);
            i = __shfl_sync(0xffffffffu, i, 0);
            if (i >= cnt) break;
            int64_t n; int32_t pb;
            const int64_t lq = first + i;
            const int64_t w0i = block_word(a.chunk0 + lq, a.W, a.rowwords, &n, &pb) - lo4;
            const int32_t p0 = pb * POS_BLOCK;
            int32_t deficit = 0;                              // warp-uniform: one row per position block
            if (RAGGED) deficit = (int32_t)(a.Lb - __ldg(a.lens + n));
            // PRMT selectors of this position block: sel[u] picks, from a column's 8 bytes {A,C,G,T}, the entries of
            // base[p0+u] (low half) and base[p0+u+1] (high half).  Same value in every lane (broadcast loads).
            uint32_t sel[NSEL];
            {
                const uint32_t* wp = s_tile + w0i;
                uint32_t wlo = wp[0];
                #pragma unroll
                for (int wi = 0; wi < (NSEL + 15) / 16; ++wi) {
                    const uint32_t whi = wp[wi + 1];
                    #pragma unroll
                    for (int uu = 0; uu < 16; ++uu) {
                        const int u = wi * 16 + uu;
                        if (u < NSEL) {
                            const uint32_t x = __funnelshift_r(wlo, whi, 2 * uu) & 15u;
                            sel[u] = 0x1010u + 0x22u * (x & 3u) + 0x2200u * (x >> 2);
                        }
                    }
                    wlo = whi;
                }
            }
            // this block is the low (pb even) or high (pb odd) half of mask word (n, pb/2)
            uint16_t* mrow = reinterpret_cast<uint16_t*>(a.mask + (lq >> 1) * (int64_t)a.K2pad + (int64_t)mbk.g0 * GROUP_SLOTS) + (pb & 1);
            uint32_t* krow = a.mask + lq * (int64_t)a.K2pad + (int64_t)mbk.g0 * GROUP_SLOTS;

            for (int32_t g = 0; g < mbk.ng; ++g) {
                const GroupMeta* gm = s_meta + g;
                if (p0 >= gm->npos_max - deficit) {           // warp-uniform: no valid start position in this block
                    if constexpr (BEST) krow[g * GROUP_SLOTS + lane] = 0u;
                    else mrow[(g * GROUP_SLOTS + lane) * 2] = 0;
                    continue;
                }
                const int32_t len = gm->len;
                const uint32_t tab = tab_base + gm->tab_off;
                __half2 acc[POS_BLOCK / 2];
                #pragma unroll
                for (int k = 0; k < POS_BLOCK / 2; ++k) acc[k] = as_h2(0u);
                // Columns are processed two per trip (tables are padded with a zero column to an even length: x + (+0) = x).
                // ptxas splits the adds between HADD2 (ALU pipe) and HFMA2(x,1,y) (FMA pipe); both round identically.
                #pragma unroll
                for (int j = 0; j < MB200_MAX_MOTIF_LEN; j += 2) {
                    if (j >= len) break;
                    const uint2 e0 = lds64(tab + j * COL_BYTES);
                    const uint2 e1 = lds64(tab + (j + 1) * COL_BYTES);
                    #pragma unroll
                    for (int k = 0; k < POS_BLOCK / 2; ++k) acc[k] = __hadd2(acc[k], as_h2(__byte_perm(e0.x, e0.y, sel[2 * k + j])));
                    #pragma unroll
                    for (int k = 0; k < POS_BLOCK / 2; ++k) acc[k] = __hadd2(acc[k], as_h2(__byte_perm(e1.x, e1.y, sel[2 * k + j + 1])));
                }
                if constexpr (BEST) {
                    // start positions past the row's last window and disabled slots (+Inf threshold: strand not requested, padding)
                    // become NaN, which __hmax2 ignores; the lowest position holding the maximum wins
                    const int32_t nvalid = gm->thr[lane] == 0x7C00u ? 0 : min(max(gm->npos[lane >> 1] - deficit - p0, 0), POS_BLOCK);
                    const uint32_t inv = ~((1u << nvalid) - 1u);
                    __half2 mx = as_h2(0x7E007E00u);
                    #pragma unroll
                    for (int k = 0; k < POS_BLOCK / 2; ++k) {
                        const uint32_t nan = ((inv >> (2 * k)) & 1u) * 0x7E00u | ((inv >> (2 * k + 1)) & 1u) * 0x7E000000u;
                        acc[k] = as_h2(*reinterpret_cast<uint32_t*>(&acc[k]) | nan);
                        mx = __hmax2(mx, acc[k]);
                    }
                    const __half m1 = __hmax(__low2half(mx), __high2half(mx));
                    const __half2 mm = __half2half2(m1);
                    uint32_t eq = 0;
                    #pragma unroll
                    for (int k = 0; k < POS_BLOCK / 2; ++k) {
                        const uint32_t m = __heq2_mask(acc[k], mm);
                        eq |= ((m & 1u) | ((m >> 15) & 2u)) << (2 * k);
                    }
                    const uint32_t u = (uint32_t)__ffs(eq) - 1u;             // eq == 0 (every position NaN): key 0
                    krow[g * GROUP_SLOTS + lane] = eq ? (h16_ord(__half_as_ushort(m1)) << 4 | (15u - u)) : 0u;
                } else {
                    const uint32_t t16 = gm->thr[lane];
                    const __half2 thr = as_h2(t16 | (t16 << 16));
                    uint32_t bits = 0;
                    #pragma unroll
                    for (int k = 0; k < POS_BLOCK / 2; ++k) {
                        const uint32_t m = __hgt2_mask(acc[k], thr);
                        bits |= ((m & 1u) | ((m >> 15) & 2u)) << (2 * k);
                    }
                    const int32_t nvalid = min(max(gm->npos[lane >> 1] - deficit - p0, 0), POS_BLOCK);
                    bits &= (1u << nvalid) - 1u;
                    mrow[(g * GROUP_SLOTS + lane) * 2] = (uint16_t)bits;
                }
            }
        }
        __syncthreads();      // tile buffer `buf` and (possibly) the blob may be overwritten next
        if (threadIdx.x == 0) s_ticket[0] = 0;
        __syncthreads();
    }
}

// Motifs longer than MB200_MAX_MOTIF_LEN columns (rare: the reference trims PWMs to their informative span) are scored by a
// plain kernel: one warp per (sequence, slot), lanes over 32 start positions, table read from global memory.  Same
// sequential Float16 adds, same mask layout.  BEST: lanes 0-15 and 16-31 reduce their starts to the best-site keys of position
// blocks 2w and 2w+1, in the key layout of scan_kernel<RAGGED, true>.
template <bool BEST = false>
__global__ void __launch_bounds__(256) scan_long_kernel(const uint32_t* __restrict__ seqw, int64_t rowwords, int64_t seq0, int64_t nseq,
                                                        int32_t W, int32_t K2pad, const uint8_t* __restrict__ blob,
                                                        const MBlock* __restrict__ lblocks, int32_t n_lblocks, uint32_t* __restrict__ mask,
                                                        const int64_t* __restrict__ lens, int64_t Lb) {
    const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int64_t per_seq = (int64_t)n_lblocks * GROUP_SLOTS;
    if (wid >= nseq * per_seq) return;
    const int64_t n = wid / per_seq;
    const int rem = (int)(wid - n * per_seq);
    const MBlock mb = lblocks[rem / GROUP_SLOTS];
    const int slot = rem % GROUP_SLOTS;
    const GroupMeta* gm = reinterpret_cast<const GroupMeta*>(blob + mb.blob_off + mb.tab_bytes);
    const uint8_t* tab = blob + mb.blob_off + slot * 8;
    const int len = gm->len;
    int npos = gm->npos[slot >> 1];
    if (lens) npos = max(0, npos - (int)(Lb - lens[seq0 + n]));          // ragged store: this row's own start positions
    const __half thr = __ushort_as_half(gm->thr[slot]);
    const uint32_t* srow = seqw + (seq0 + n) * rowwords;
    if (BEST && gm->thr[slot] == 0x7C00u) npos = 0;                     // strand not requested
    for (int w = 0; w < W; ++w) {
        const int pos = w * 32 + lane;
        bool hit = false;
        uint32_t key = 0;
        if (pos < npos) {
            __half s = __ushort_as_half((unsigned short)0);
            for (int j = 0; j < len; ++j) {
                const int q = pos + j;
                const uint32_t base = (srow[q >> 4] >> ((q & 15) * 2)) & 3u;
                s = __hadd(s, *reinterpret_cast<const __half*>(tab + (int64_t)j * COL_BYTES + base * 2));
            }
            hit = __hgt(s, thr);
            if (BEST && !__hisnan(s)) key = h16_ord(__half_as_ushort(s)) << 4 | (15u - (uint32_t)(lane & 15));
        }
        if constexpr (BEST) {
            #pragma unroll
            for (int o = 8; o >= 1; o >>= 1) key = max(key, __shfl_xor_sync(0xffffffffu, key, o));
            if ((lane & 15) == 0) mask[(n * 2 * W + 2 * w + (lane >> 4)) * (int64_t)K2pad + (int64_t)mb.g0 * GROUP_SLOTS + slot] = key;
        } else {
            const uint32_t word = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) mask[(n * W + w) * (int64_t)K2pad + (int64_t)mb.g0 * GROUP_SLOTS + slot] = word;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Best site per (row, motif) from the block keys of scan_kernel<RAGGED, true> / scan_long_kernel<true>: one thread per (row,
// motif, chunk of <= BEST_CHUNK position blocks); adjacent threads take adjacent motifs, so the (fwd, rc) key pairs load
// coalesced.  A thread's best goes into best64[row * K + motif] by atomicMax on
//   ord(score) << 48 | (0xFFFFFFFF - pos) << 1 | (1 - comp)
// (higher score, then lower position, then the forward strand), a total order: the result does not depend on the order of
// arrival.  0 = no window.
// ---------------------------------------------------------------------------------------------
#define BEST_CHUNK 1024
__global__ void __launch_bounds__(256) best_reduce_kernel(const uint32_t* __restrict__ keys, int64_t nseq, int32_t W16, int32_t K2pad, int32_t nch,
                                                          const int32_t* __restrict__ pair2motif, int32_t K, unsigned long long* __restrict__ best64) {
    const int32_t P = K2pad / 2;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nseq * nch * P) return;
    const int32_t m2 = (int32_t)(t % P);
    const int64_t nc = t / P;
    const int32_t c = (int32_t)(nc % nch);
    const int64_t n = nc / nch;
    const int32_t k = pair2motif[m2];
    if (k < 0) return;
    const uint2* kp = reinterpret_cast<const uint2*>(keys) + (n * W16) * (int64_t)P + m2;
    const int32_t b0 = c * BEST_CHUNK, b1 = min(W16, b0 + BEST_CHUNK);
    unsigned long long best = 0;
    for (int32_t b = b0; b < b1; ++b) {
        const uint2 fr = __ldg(kp + (int64_t)b * P);
        if (fr.x) best = max(best, (unsigned long long)(fr.x >> 4) << 48 | (unsigned long long)(0xFFFFFFFFu - (uint32_t)(b * POS_BLOCK + 15 - (fr.x & 15u))) << 1 | 1ull);
        if (fr.y) best = max(best, (unsigned long long)(fr.y >> 4) << 48 | (unsigned long long)(0xFFFFFFFFu - (uint32_t)(b * POS_BLOCK + 15 - (fr.y & 15u))) << 1);
    }
    if (best) atomicMax(best64 + n * K + k, best);
}

__global__ void __launch_bounds__(256) best_finalize_kernel(const unsigned long long* __restrict__ best64, int64_t n, mb200_best* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long v = best64[i];
    mb200_best r;
    if (v) {
        const uint32_t o = (uint32_t)(v >> 48);
        r.pos = 0xFFFFFFFFu - (uint32_t)(v >> 1);
        r.score_f16 = (uint16_t)((o & 0x8000u) ? (o & 0x7FFFu) : (~o & 0xFFFFu));
        r.comp = (uint8_t)(1u - (uint32_t)(v & 1u));
        r.found = 1;
    } else {
        r.pos = 0xFFFFFFFFu; r.score_f16 = 0; r.comp = 0; r.found = 0;
    }
    out[i] = r;
}

// ---------------------------------------------------------------------------------------------
// Spacing mode (mb200_scan_spacing): rows 2i and 2i + 1 of the scanned store are the left and right margins of anchor i, and
// best64 holds their best-site keys.  One thread per (anchor, secondary), adjacent threads on adjacent secondaries (the key loads
// coalesce).  The two margins merge by score alone: on equal scores the left margin's window lies lower in the row.  A counted
// window (score > thr[k], with thr = max(thresh, 0) and +Inf for a NaN threshold, as build_plan sets them) adds 1 to its
// (primary, k, quadrant, gap) bin; integer atomics make the histogram independent of the order of arrival.
// ---------------------------------------------------------------------------------------------
static_assert(sizeof(mb200_anchor) == 24, "mb200_anchor must be 24 bytes");
__global__ void __launch_bounds__(256) spacing_kernel(const unsigned long long* __restrict__ best64, int64_t na, int32_t K,
                                                      const mb200_anchor* __restrict__ anchors, const uint16_t* __restrict__ thr,
                                                      const int32_t* __restrict__ mlen, int32_t margin, unsigned int* __restrict__ hist,
                                                      mb200_best* __restrict__ sites) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= na * K) return;
    const int64_t i = t / K;
    const int32_t k = (int32_t)(t - i * K);
    const unsigned long long l = best64[2 * i * K + k], r = best64[(2 * i + 1) * K + k];
    const bool left = l && (l >> 48) >= (r >> 48);
    const unsigned long long v = left ? l : r;
    mb200_best out;
    out.pos = 0xFFFFFFFFu; out.score_f16 = 0; out.comp = 0; out.found = 0;
    if (v) {
        const mb200_anchor an = anchors[i];
        const uint32_t o = (uint32_t)(v >> 48);
        const uint16_t s = (uint16_t)((o & 0x8000u) ? (o & 0x7FFFu) : (~o & 0xFFFFu));
        const int32_t u = (int32_t)(0xFFFFFFFFu - (uint32_t)(v >> 1));          // start inside the margin
        const uint32_t c = 1u - (uint32_t)(v & 1u);
        const bool counted = __hgt(__ushort_as_half(s), __ushort_as_half(thr[k]));
        out.pos = (uint32_t)(left ? an.start - margin + u : an.start + an.len + u);
        out.score_f16 = s; out.comp = (uint8_t)c; out.found = counted;
        if (counted) {
            const int32_t g = left ? margin - u - mlen[k] : u;
            const int32_t down = left == (an.comp != 0);
            const int32_t q = 2 * (int32_t)(c != an.comp) + down;
            atomicAdd(hist + (((int64_t)an.primary * K + k) * 4 + q) * margin + g, 1u);
        }
    }
    if (sites) sites[t] = out;
}

// what mb200_scan_spacing hands to scan_impl: host arrays
struct SpacingJob {
    const mb200_anchor* anchors; int64_t n;
    int32_t n_primary, margin;
    const uint16_t* thresh;            // K Float16 bits or NULL
    uint32_t* hist;                    // n_primary * K * 4 * margin
    mb200_best* sites;                 // n * K or NULL
};

// ---------------------------------------------------------------------------------------------
// Counting from the masks: one thread per (sequence, motif).  Mask word layout:
//   mask[(n*W + w) * K2pad + slotpair*2 + strand]
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t dilate32(uint32_t u, int len) {
    // set bits i..i+len-1 for every set bit i (bits above 31 are dropped)
    uint32_t r = u; int k = 1;
    while (k < len && k < 32) { int s = min(k, len - k); r |= r << s; k += s; }
    return r;
}

// counts of one (sequence, motif) unit from its W mask words of both strands; CLEAR: leave the words zero behind (the tensor-core
// path keeps the mask buffer all-zero between batches instead of clearing 8 GB per batch)
template <bool CLEAR>
__device__ __forceinline__ void count_unit(uint32_t* __restrict__ mask, int64_t n, int32_t m2, int32_t W, int32_t P, int32_t k, int32_t len,
                                           unsigned long long* __restrict__ counts, uint32_t* __restrict__ unit_cnt, int32_t K) {
    uint2* mp = reinterpret_cast<uint2*>(mask) + (n * W) * (int64_t)P + m2;
    uint32_t nf = 0, nr = 0, uq = 0, cov = 0;
    int32_t cu = 0;             // positions < cu are covered by earlier hits
    int32_t p1 = -1, p2 = -1;   // largest / second largest distinct start position
    bool dup = false;           // p1 hit on both strands
    for (int32_t w = 0; w < W; ++w) {
        const uint2 fr = CLEAR ? mp[(int64_t)w * P] : __ldg(mp + (int64_t)w * P);
        const uint32_t f = fr.x, r = fr.y, U = f | r;
        const int32_t base = w * 32;
        const int32_t cb = cu - base;
        uint32_t cm = cb >= 32 ? 0xffffffffu : (cb > 0 ? ((1u << cb) - 1u) : 0u);
        if (U) {
            if (CLEAR) mp[(int64_t)w * P] = make_uint2(0u, 0u);
            nf += __popc(f); nr += __popc(r); uq += __popc(U);
            cm |= dilate32(U, len);
            const int32_t hi = 31 - __clz(U);
            cu = max(cu, base + hi + len);
            const uint32_t U2 = U & ~(1u << hi);
            p2 = U2 ? base + 31 - __clz(U2) : p1;
            p1 = base + hi;
            dup = ((f >> hi) & (r >> hi) & 1u) != 0;
        }
        cov += __popc(cm);
    }
    cov += max(0, cu - W * 32);
    const uint32_t nh = nf + nr;
    if (unit_cnt) {
        reinterpret_cast<uint2*>(unit_cnt)[n * K + k] = make_uint2(nf, nr);
    }
    if (nh) {
        uint32_t covq = cov;
        if (nh >= 2 && !dup) covq -= (uint32_t)min(len, p1 - p2);   // union_ranges drops the last interval
        atomicAdd(&counts[k * 4 + 0], (unsigned long long)nh);
        atomicAdd(&counts[k * 4 + 1], (unsigned long long)uq);
        atomicAdd(&counts[k * 4 + 2], (unsigned long long)covq);
        atomicAdd(&counts[k * 4 + 3], (unsigned long long)cov);
    }
}

__global__ void __launch_bounds__(256) count_kernel(const uint32_t* __restrict__ mask, int64_t nseq, int32_t W, int32_t K2pad,
                                                    const int32_t* __restrict__ pair2motif, const int32_t* __restrict__ pairlen,
                                                    unsigned long long* __restrict__ counts, uint32_t* __restrict__ unit_cnt, int32_t K) {
    const int32_t P = K2pad / 2;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nseq * P) return;
    const int64_t n = t / P;
    const int32_t m2 = (int32_t)(t - n * P);
    const int32_t k = pair2motif[m2];
    if (k < 0) return;
    count_unit<false>(const_cast<uint32_t*>(mask), n, m2, W, P, k, pairlen[m2], counts, unit_cnt, K);
}

// Sparse form for the tensor-core path: one thread per (sequence, motif) unit that received at least one hit (the verifier lists
// them); all other units have no hits and contribute nothing.  Clears the words it reads.
__global__ void __launch_bounds__(256) count_listed_kernel(uint32_t* __restrict__ mask, const uint32_t* __restrict__ units, const unsigned long long* __restrict__ n_units,
                                                           int32_t W, int32_t K2pad, const int32_t* __restrict__ pair2motif, const int32_t* __restrict__ pairlen,
                                                           unsigned long long* __restrict__ counts, const unsigned long long* __restrict__ overflow,
                                                           uint32_t* __restrict__ unit_cnt, int32_t K, int32_t clear) {
    const int32_t P = K2pad / 2;
    if (overflow && *overflow) return;                                                    // candidate list overflowed: the batch is re-run on scan_kernel
    const unsigned long long total = *n_units;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t g = units[i];
        const int64_t n = g / (uint32_t)P;
        const int32_t m2 = (int32_t)(g - (uint32_t)n * (uint32_t)P);
        if (clear) count_unit<true>(mask, n, m2, W, P, pair2motif[m2], pairlen[m2], counts, unit_cnt, K);
        else count_unit<false>(mask, n, m2, W, P, pair2motif[m2], pairlen[m2], counts, unit_cnt, K);     // the hit list is still to be emitted from these words
    }
}
// after the hit list has been emitted: zero the mask words of the listed units so that the buffer is all-zero again
__global__ void __launch_bounds__(256) clear_listed_kernel(uint32_t* __restrict__ mask, const uint32_t* __restrict__ units, const unsigned long long* __restrict__ n_units,
                                                           int32_t W, int32_t K2pad) {
    const int32_t P = K2pad / 2;
    const unsigned long long total = *n_units * (unsigned long long)W;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t g = units[i / W];
        const int32_t w = (int32_t)(i % W);
        const int64_t n = g / (uint32_t)P;
        const int32_t m2 = (int32_t)(g - (uint32_t)n * (uint32_t)P);
        reinterpret_cast<uint2*>(mask)[((n * W) + w) * (int64_t)P + m2] = make_uint2(0u, 0u);
    }
}


// ---------------------------------------------------------------------------------------------
// Counting for long sequences (chromosome-scale, BASELINE config 5): the W mask words of a sequence are cut into blocks of
// WB words so that one thread per (sequence, block, motif) runs in parallel.  Coverage needs only a short look-back (a hit
// reaches at most len-1 positions forward); the union_ranges quirk needs the two largest distinct start positions of the whole
// sequence, found with two rounds of atomicMax.
// ---------------------------------------------------------------------------------------------
struct LongCand { int32_t p1, p2, dup; };

__global__ void __launch_bounds__(256) count_long_a(const uint32_t* __restrict__ mask, int64_t nseq, int32_t W, int32_t K2pad, int32_t WB, int32_t nblocks,
                                                    const int32_t* __restrict__ pair2motif, const int32_t* __restrict__ pairlen,
                                                    unsigned long long* __restrict__ counts, unsigned long long* __restrict__ top1,
                                                    unsigned int* __restrict__ nh_seq, LongCand* __restrict__ cand) {
    const int32_t P = K2pad / 2;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nseq * nblocks * P) return;
    const int32_t m2 = (int32_t)(t % P);
    const int64_t nb = t / P;
    const int32_t wb = (int32_t)(nb % nblocks);
    const int64_t n = nb / nblocks;
    LongCand c; c.p1 = -1; c.p2 = -1; c.dup = 0;
    const int32_t k = pair2motif[m2];
    if (k >= 0) {
        const int32_t len = pairlen[m2];
        const uint2* mp = reinterpret_cast<const uint2*>(mask) + (n * W) * (int64_t)P + m2;
        const int32_t w0 = wb * WB, w1 = min(W, w0 + WB);
        int32_t cu = 0;
        const int32_t LB = (len + 31) / 32 + 1;
        for (int32_t w = w0 - 1; w >= max(0, w0 - LB); --w) {           // nearest earlier hit decides the carried coverage
            const uint2 fr = __ldg(mp + (int64_t)w * P);
            const uint32_t U = fr.x | fr.y;
            if (U) { cu = w * 32 + 31 - __clz(U) + len; break; }
        }
        uint32_t nf = 0, nr = 0, uq = 0; unsigned long long cov = 0;
        for (int32_t w = w0; w < w1; ++w) {
            const uint2 fr = __ldg(mp + (int64_t)w * P);
            const uint32_t f = fr.x, r = fr.y, U = f | r;
            const int32_t base = w * 32;
            const int32_t cb = cu - base;
            uint32_t cm = cb >= 32 ? 0xffffffffu : (cb > 0 ? ((1u << cb) - 1u) : 0u);
            if (U) {
                nf += __popc(f); nr += __popc(r); uq += __popc(U);
                cm |= dilate32(U, len);
                const int32_t hi = 31 - __clz(U);
                cu = max(cu, base + hi + len);
                const uint32_t U2 = U & ~(1u << hi);
                c.p2 = U2 ? base + 31 - __clz(U2) : c.p1;
                c.p1 = base + hi;
                c.dup = ((f >> hi) & (r >> hi) & 1u) != 0;
            }
            cov += __popc(cm);
        }
        if (w1 == W) cov += (unsigned long long)max(0, cu - W * 32);   // positions covered past the last mask word
        const uint32_t nh = nf + nr;
        if (nh) {
            atomicAdd(&counts[k * 4 + 0], (unsigned long long)nh);
            atomicAdd(&counts[k * 4 + 1], (unsigned long long)uq);
            atomicAdd(&nh_seq[n * P + m2], nh);
            atomicMax(&top1[n * P + m2], (unsigned long long)(c.p1 + 1));
        }
        if (cov) { atomicAdd(&counts[k * 4 + 2], cov); atomicAdd(&counts[k * 4 + 3], cov); }
    }
    cand[t] = c;
}
__global__ void __launch_bounds__(256) count_long_b(int64_t nseq, int32_t P, int32_t nblocks, const LongCand* __restrict__ cand,
                                                    const unsigned long long* __restrict__ top1, unsigned long long* __restrict__ top2,
                                                    unsigned int* __restrict__ dupflag) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nseq * nblocks * P) return;
    const int32_t m2 = (int32_t)(t % P);
    const int64_t n = (t / P) / nblocks;
    const LongCand c = cand[t];
    if (c.p1 < 0) return;
    const long long g1 = (long long)top1[n * P + m2] - 1;
    int32_t second;
    if (c.p1 == g1) { second = c.p2; if (c.dup) dupflag[n * P + m2] = 1u; } else second = c.p1;
    if (second >= 0) atomicMax(&top2[n * P + m2], (unsigned long long)(second + 1));
}
__global__ void __launch_bounds__(256) count_long_c(int64_t nseq, int32_t P, const int32_t* __restrict__ pair2motif, const int32_t* __restrict__ pairlen,
                                                    const unsigned long long* __restrict__ top1, const unsigned long long* __restrict__ top2,
                                                    const unsigned int* __restrict__ dupflag, const unsigned int* __restrict__ nh_seq,
                                                    unsigned long long* __restrict__ counts) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nseq * P) return;
    const int32_t m2 = (int32_t)(t % P);
    const int32_t k = pair2motif[m2];
    if (k < 0 || nh_seq[t] < 2 || dupflag[t]) return;
    const long long p1 = (long long)top1[t] - 1, p2 = (long long)top2[t] - 1;
    const long long drop = min((long long)pairlen[m2], p1 - p2);           // union_ranges never visits the last sorted interval
    atomicAdd(&counts[k * 4 + 2], (unsigned long long)(-drop));
}

// ---------------------------------------------------------------------------------------------
// Exclusive prefix sum u32 -> u64 (three small kernels), used to place hits without atomics.
// ---------------------------------------------------------------------------------------------
#define PS_THREADS 256
#define PS_ITEMS 8
#define PS_TILE (PS_THREADS * PS_ITEMS)

__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long* total) {
    __shared__ unsigned long long s_w[PS_THREADS / 32 + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long inc = v;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { unsigned long long y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        unsigned long long x = lane < (int)(blockDim.x >> 5) ? s_w[lane] : 0ull, xi = x;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) { unsigned long long y = __shfl_up_sync(0xffffffffu, xi, o); if (lane >= o) xi += y; }
        if (lane < (int)(blockDim.x >> 5)) s_w[lane] = xi - x;
        if (lane == 31) s_w[PS_THREADS / 32] = xi;
    }
    __syncthreads();
    unsigned long long r = s_w[warp] + inc - v;
    if (total) *total = s_w[PS_THREADS / 32];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(PS_THREADS) ps_block_sums(const uint32_t* __restrict__ in, int64_t n, unsigned long long* __restrict__ bsum) {
    const int64_t base = (int64_t)blockIdx.x * PS_TILE;
    unsigned long long s = 0;
    #pragma unroll
    for (int i = 0; i < PS_ITEMS; ++i) { int64_t j = base + (int64_t)i * PS_THREADS + threadIdx.x; if (j < n) s += in[j]; }
    unsigned long long tot;
    block_excl_scan(s, &tot);
    if (threadIdx.x == 0) bsum[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(PS_THREADS) ps_scan_sums(unsigned long long* __restrict__ bsum, int64_t nb, unsigned long long* __restrict__ total) {
    unsigned long long carry = 0;
    for (int64_t b0 = 0; b0 < nb; b0 += PS_THREADS) {
        int64_t j = b0 + threadIdx.x;
        unsigned long long v = j < nb ? bsum[j] : 0ull, tot;
        unsigned long long e = block_excl_scan(v, &tot);
        if (j < nb) bsum[j] = carry + e;
        carry += tot;
    }
    if (threadIdx.x == 0) *total = carry;
}
__global__ void __launch_bounds__(PS_THREADS) ps_apply(const uint32_t* __restrict__ in, int64_t n, const unsigned long long* __restrict__ bsum,
                                                       unsigned long long* __restrict__ out) {
    const int64_t base = (int64_t)blockIdx.x * PS_TILE + (int64_t)threadIdx.x * PS_ITEMS;
    uint32_t v[PS_ITEMS]; unsigned long long s = 0;
    #pragma unroll
    for (int i = 0; i < PS_ITEMS; ++i) { v[i] = (base + i < n) ? in[base + i] : 0u; s += v[i]; }
    unsigned long long e = block_excl_scan(s, nullptr) + bsum[blockIdx.x];
    #pragma unroll
    for (int i = 0; i < PS_ITEMS; ++i) { if (base + i < n) out[base + i] = e; e += v[i]; }
}

// ---------------------------------------------------------------------------------------------
// Hit emission: one thread per (sequence, motif, strand) walks its mask bits in ascending position
// and recomputes the Float16 score with the same sequential adds as the scan kernel.
// ---------------------------------------------------------------------------------------------
// slot = global mask slot of the forward strand; tab_off = byte offset (in the blob) of the forward entry (column 0, base A)
struct EmitMotif { int32_t slot; int32_t len; int64_t tab_off; int32_t col_stride, base_stride, strand_stride, pad; };

__global__ void __launch_bounds__(256) emit_kernel(const uint32_t* __restrict__ mask, const uint32_t* __restrict__ seqw, int64_t rowwords,
                                                   int64_t seq0, int64_t nseq, int32_t W, int32_t K2pad, int32_t K,
                                                   const EmitMotif* __restrict__ em, const uint8_t* __restrict__ blob,
                                                   const uint32_t* __restrict__ unit_cnt, const unsigned long long* __restrict__ unit_off,
                                                   mb200_hit* __restrict__ hits) {
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nseq * K * 2) return;
    if (unit_cnt[u] == 0) return;
    const int32_t strand = (int32_t)(u & 1);
    const int64_t nk = u >> 1;
    const int64_t n = nk / K;
    const int32_t k = (int32_t)(nk - n * K);
    const EmitMotif m = em[k];
    const int32_t slot = m.slot + strand;
    const uint8_t* tab = blob + m.tab_off + strand * m.strand_stride;
    const uint32_t* srow = seqw + (seq0 + n) * rowwords;
    unsigned long long off = unit_off[u];
    for (int32_t w = 0; w < W; ++w) {
        uint32_t bits = mask[((n * W) + w) * (int64_t)K2pad + slot];
        while (bits) {
            const int32_t b = __ffs(bits) - 1;
            bits &= bits - 1;
            const int32_t p = w * 32 + b;
            __half s = __ushort_as_half((unsigned short)0);
            for (int32_t j = 0; j < m.len; ++j) {
                const int32_t q = p + j;
                const uint32_t base = (srow[q >> 4] >> ((q & 15) * 2)) & 3u;
                const __half e = *reinterpret_cast<const __half*>(tab + (int64_t)j * m.col_stride + base * m.base_stride);
                s = __hadd(s, e);
            }
            // mb200_hit as one 16 B store: {seq, pos, motif | score<<16, comp}
            const uint4 h = make_uint4((uint32_t)(seq0 + n), (uint32_t)p,
                                       (uint32_t)k | ((uint32_t)__half_as_ushort(s) << 16), (uint32_t)strand);
            reinterpret_cast<uint4*>(hits)[off++] = h;
        }
    }
}


// Score histogram (SURVEY §8f-1): for every hit the Float16 score is recomputed as in emit_kernel and counted in
// hist[motif][score bits] (positive halves order like their 15-bit patterns).  Feeds the threshold sweep of get_best_thresh
// (inference/_s2_filter_pos_w_scores.jl:99-113: hits with score > t for t = min_score : 0.5 : max_score) without building hit lists.
#define HIST_BINS 32768
__global__ void __launch_bounds__(256) hist_kernel(const uint32_t* __restrict__ mask, const uint32_t* __restrict__ seqw, int64_t rowwords,
                                                   int64_t seq0, int64_t nseq, int32_t W, int32_t K2pad, int32_t K,
                                                   const EmitMotif* __restrict__ em, const uint8_t* __restrict__ blob, unsigned int* __restrict__ hist) {
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nseq * K * 2) return;
    const int32_t strand = (int32_t)(u & 1);
    const int64_t nk = u >> 1;
    const int64_t n = nk / K;
    const int32_t k = (int32_t)(nk - n * K);
    const EmitMotif m = em[k];
    const int32_t slot = m.slot + strand;
    const uint8_t* tab = blob + m.tab_off + strand * m.strand_stride;
    const uint32_t* srow = seqw + (seq0 + n) * rowwords;
    for (int32_t w = 0; w < W; ++w) {
        uint32_t bits = mask[((n * W) + w) * (int64_t)K2pad + slot];
        while (bits) {
            const int32_t b = __ffs(bits) - 1;
            bits &= bits - 1;
            const int32_t p = w * 32 + b;
            __half s = __ushort_as_half((unsigned short)0);
            for (int32_t j = 0; j < m.len; ++j) {
                const int32_t q = p + j;
                const uint32_t base = (srow[q >> 4] >> ((q & 15) * 2)) & 3u;
                s = __hadd(s, *reinterpret_cast<const __half*>(tab + (int64_t)j * m.col_stride + base * m.base_stride));
            }
            atomicAdd(&hist[(int64_t)k * HIST_BINS + (__half_as_ushort(s) & 0x7FFFu)], 1u);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Host side: plan (sorted groups, tables, thresholds), batching, launches.
// ---------------------------------------------------------------------------------------------
static inline bool h16_nonfinite(uint16_t h) { return (h & 0x7C00u) == 0x7C00u; }
static inline float h16_to_float(uint16_t h) { __half_raw r; r.x = h; return __half2float(__half(r)); }
// The hit rule: a window hits when its Float16 score > max(thresh[k], 0), and never for a NaN threshold.  Returns the Float16 bits
// of that effective threshold: 0x7C00 (+Inf) for a NaN threshold, 0 without thresholds.
static uint16_t hit_threshold(const uint16_t* thresh, int k) {
    if (!thresh) return 0;
    const uint16_t raw = thresh[k];
    if (h16_nonfinite(raw) && (raw & 0x03FFu)) return 0x7C00u;
    return h16_to_float(raw) > 0.f ? raw : (uint16_t)0;
}

struct ScanPlan {
    int K = 0, ngroups = 0, K2pad = 0;
    std::vector<uint8_t> blob;
    std::vector<MBlock> mblocks;
    std::vector<MBlock> lblocks;          // one per group of motifs longer than MB200_MAX_MOTIF_LEN (slow path)
    std::vector<int32_t> pair2motif, pairlen;
    std::vector<EmitMotif> em;
    int max_blob_bytes = 0;
    int minlen = 0;
};

#include "scan_tc.cuh"

// ---- host side of the tensor-core pre-filter (scan_tc.cuh) ------------------------------------------------------------
static inline uint16_t float_to_h16(float f) { __half h = __float2half_rn(f); __half_raw r = h; return r.x; }
static inline uint16_t h16_nextup(uint16_t h) { if (h == 0x8000u) return 0x0001u; return (h & 0x8000u) ? (uint16_t)(h - 1) : (uint16_t)(h + 1); }
// smallest Float16 >= x (|x| well inside the Float16 range)
static inline uint16_t h16_round_up(double x) {
    uint16_t h = float_to_h16((float)x);
    while ((double)h16_to_float(h) < x) h = h16_nextup(h);
    return h;
}
// E with |Float16 running sum - real sum| <= E for every path through the columns w[j][0..3] whose Float16 running sum ends above t.
//   U_j = fl16(U_{j-1} + max_b w[j][b])  bounds every partial sum from above (rounding is monotone);
//   for paths ending above t:  s_{j-1} >= L_{j-1} = L_j - max_b w[j][b] - u*B_j,  L_n = t,  B_j = max(|L_j|, |U_j|) >= |s_j|;
//   each add errs by at most u*|s_j|, u = 2^-11 (results in the subnormal range are exact).  Returns false when U_n <= t (no hit possible).
static bool tc_error_bound(const std::vector<double>& w, int n, double t, double* E_out) {
    const double u = 1.0 / 2048.0;
    std::vector<double> U(n + 1, 0.0), mx(n + 1, 0.0);
    for (int j = 1; j <= n; ++j) {
        double m = w[(size_t)(j - 1) * 4];
        for (int b = 1; b < 4; ++b) m = std::max(m, w[(size_t)(j - 1) * 4 + b]);
        mx[j] = m;
        U[j] = (double)h16_to_float(float_to_h16((float)(U[j - 1] + m)));     // the sum of two halves is exact in float: one rounding
    }
    if (!(U[n] > t)) return false;
    double L = t, E = 0.0;
    for (int j = n; j >= 1; --j) {
        const double B = std::max(std::fabs(L), std::fabs(U[j]));
        E += u * B;
        L = L - mx[j] - u * B;
    }
    *E_out = E * 1.001 + 1e-6;
    return true;
}

// CTAs of the grid over slot blocks in proportion to cost (clocks per tile); every block gets at least one.
static bool tc_assign_ctas(std::vector<TcBlock>& blocks, const std::vector<double>& cost, int grid) {
    const int nblocks = (int)blocks.size();
    if (nblocks > grid) return false;
    double csum = 0; for (double c : cost) csum += c;
    std::vector<int> n(nblocks);
    int used = 0;
    for (int bi = 0; bi < nblocks; ++bi) { n[bi] = std::max(1, (int)(grid * cost[bi] / csum)); used += n[bi]; }
    while (used > grid) {                                         // take from the block with the least cost per CTA
        int w = -1;
        for (int bi = 0; bi < nblocks; ++bi) if (n[bi] > 1 && (w < 0 || cost[bi] / n[bi] < cost[w] / n[w])) w = bi;
        if (w < 0) return false;
        --n[w]; --used;
    }
    while (used < grid) {                                         // give to the block with the most cost per CTA
        int w = 0;
        for (int bi = 1; bi < nblocks; ++bi) if (cost[bi] / n[bi] > cost[w] / n[w]) w = bi;
        ++n[w]; ++used;
    }
    int c0 = 0;
    for (int bi = 0; bi < nblocks; ++bi) { blocks[bi].cta0 = c0; blocks[bi].nctas = n[bi]; c0 += n[bi]; }
    return true;
}

// Pre-filter threshold of one slot: T' = t - E - eps32, eps32 for the FP32 accumulation in the tensor core (operands exact, possibly
// truncating adds, subnormal operands possibly flushed).  A = sum over columns of the largest |entry|.
static bool tc_prefilter_threshold(const std::vector<double>& w, int len, double t, double A, double* E_out, double* Tp_out) {
    double E = 0.0;
    if (!tc_error_bound(w, len, t, &E)) return false;
    const double eps32 = (A + std::fabs(t) + E) * (1.0 / 8192.0) + len * 6.2e-5;
    *E_out = E; *Tp_out = t - E - eps32;
    return true;
}

// The exact integer form of a slot's filter, which the tensor core evaluates.  f: the real-valued filter [len][4] (Float16 values:
// column 0 = w_0 - T' rounded up, then w_1 ..), D_real = sum_j f[j][x_j]; every true hit has D_real > eps32 > 0.
//   Q[j][b] = ceil(2^e f[j][b]) + k[j],  sum_j k[j] = 0,  Q in [-128, 127]
// 2^e f is exact (a power-of-two multiple of a Float16), so nothing is rounded down and sum_j Q[j][x_j] >= 2^e D_real for every
// window: a true hit gives an integer >= 1 and the candidate test stays D > 0.  Int32 accumulation of |Q| <= 128 x 64 is exact.
// An entry c with c + (the largest sum of the other columns) <= 0 never takes part in a positive window; it is raised to that bound
// (raising keeps the inequality, and such windows stay <= 0), so that log-odds near -Inf do not force a small scale.  The offsets
// k move column 0's large -T' term across the columns so that each fits the int8 range.  The largest e that fits has the finest
// resolution and so the fewest candidates (the rounding up loosens the filter by < len / 2^e).  Returns e.
static int tc_int8_filter(const std::vector<double>& f, int len, int8_t* Q, int32_t* k) {
    std::vector<int64_t> c((size_t)len * 4), hi(len), lo(len);
    for (int e = 24;; --e) {
        const double s = std::ldexp(1.0, e);
        int64_t H = 0;
        for (int j = 0; j < len; ++j) {
            hi[j] = INT64_MIN;
            for (int b = 0; b < 4; ++b) { c[(size_t)j * 4 + b] = (int64_t)std::ceil(s * f[(size_t)j * 4 + b]); hi[j] = std::max(hi[j], c[(size_t)j * 4 + b]); }
            H += hi[j];
        }
        bool fits = H <= 127ll * len;
        int64_t L = 0;
        for (int j = 0; j < len && fits; ++j) {
            lo[j] = INT64_MAX;
            for (int b = 0; b < 4; ++b) {
                int64_t& x = c[(size_t)j * 4 + b];
                x = std::max(x, std::min(hi[j], hi[j] - H));       // the other columns sum to at most H - hi[j]
                lo[j] = std::min(lo[j], x);
            }
            fits = hi[j] - lo[j] <= 255;
            L += lo[j];
        }
        if (!fits || L < -128ll * len) continue;                   // e = -24 always fits: every entry is then 0 or 1
        // k[j] in [-128 - lo[j], 127 - hi[j]]: start at the lower ends (sum -128 len - L <= 0) and raise them to a zero sum
        int64_t R = 128ll * len + L;
        for (int j = 0; j < len; ++j) {
            const int64_t d = std::min<int64_t>(255 - (hi[j] - lo[j]), R);
            k[j] = (int32_t)(-128 - lo[j] + d); R -= d;
            for (int b = 0; b < 4; ++b) Q[(size_t)j * 4 + b] = (int8_t)(c[(size_t)j * 4 + b] + k[j]);
        }
        return e;
    }
}

struct TcPlan {
    std::vector<uint8_t> blob;
    std::vector<TcBlock> blocks;
    std::vector<TcSlot> slots;
    size_t max_b_bytes = 0;                // largest B operand footprint of an entry
    std::vector<double> cost;              // clocks per tile of every entry (model, then measured)
};

// false: this call is not eligible for the tensor-core path (the caller keeps scan_kernel).
static bool build_tc_plan(const ScanPlan& P, const uint16_t* pwms, const int64_t* lens, int K, const uint16_t* thresh, uint32_t flags,
                          int64_t Lb, int grid, TcPlan& T) {
    if (!thresh || !P.lblocks.empty()) return false;
    const int nslots = (P.K2pad + TCS_N - 1) / TCS_N * TCS_N;
    const int nblocks = nslots / TCS_N;
    if (nblocks > grid || nblocks > TCS_MAX_ENTRIES) return false;
    auto pw = [&](int k, int a, int ind) -> uint16_t { return pwms[(size_t)k + (size_t)K * ((size_t)a + 4 * (size_t)ind)]; };
    TcSlot off; memset(&off, 0, sizeof off); off.motif = -1; off.thr = 0x7C00u;
    T.slots.assign(nslots, off);
    std::vector<std::vector<int8_t>> tab(nslots);                 // per slot: the B entries [len][4] (tc_int8_filter)
    std::vector<int> blen(nblocks, 0);
    for (int k = 0; k < K; ++k) {
        const int len = (int)lens[k];
        if (len > MB200_MAX_MOTIF_LEN) return false;
        bool neg_inf = false;
        for (int j = 0; j < len; ++j)
            for (int b = 0; b < 4; ++b) {
                const uint16_t v = pw(k, b, j);
                if (h16_nonfinite(v)) { if (v == 0xFC00u) neg_inf = true; else return false; }     // +Inf / NaN entries: leave it to scan_kernel
            }
        const uint16_t tb = hit_threshold(thresh, k);
        if (tb == 0x7C00u) continue;                               // NaN or +Inf threshold: never a hit
        const double t = (double)h16_to_float(tb);
        if (neg_inf) continue;                                     // a -Inf entry makes every window -Inf or NaN (0 * -Inf): never a hit
        for (int strand = 0; strand < 2; ++strand) {
            if (!(flags & (strand ? MB200_SCAN_RC : MB200_SCAN_FWD))) continue;
            const int slot = P.em[k].slot + strand;
            std::vector<double> w((size_t)len * 4);
            double A = 0.0;
            for (int j = 0; j < len; ++j) {
                double am = 0.0;
                for (int b = 0; b < 4; ++b) {
                    const uint16_t v = strand ? pw(k, 3 - b, len - 1 - j) : pw(k, b, j);
                    w[(size_t)j * 4 + b] = (double)h16_to_float(v);
                    am = std::max(am, std::fabs(w[(size_t)j * 4 + b]));
                }
                A += am;
            }
            double E = 0.0, Tp = 0.0;
            if (!tc_prefilter_threshold(w, len, t, A, &E, &Tp)) continue;       // the best window cannot exceed the threshold
            if (A + std::fabs(Tp) > 30000.0) return false;
            TcSlot sl; memset(&sl, 0, sizeof sl);
            sl.motif = k; sl.strand = strand; sl.len = len; sl.npos = (int32_t)std::max<int64_t>(0, Lb - len + 1); sl.thr = tb;
            T.slots[slot] = sl;
            std::vector<double> f(w);
            for (int b = 0; b < 4; ++b) f[b] = (double)h16_to_float(h16_round_up(w[b] - Tp));   // D_real > 0  <=>  real sum > T' (or a little less)
            std::vector<int32_t> koff(len);
            tab[slot].resize((size_t)len * 4);
            tc_int8_filter(f, len, tab[slot].data(), koff.data());
            blen[slot / TCS_N] = std::max(blen[slot / TCS_N], len);
        }
    }
    // B operands: [block][kchunk][256 slots][16 int8]; byte e of chunk c = column 4c + e/4, base e%4
    size_t total = 0;
    std::vector<int> kcs(nblocks);
    std::vector<int64_t> boff(nblocks);
    auto bbytes_of = [&](int kc) { return (size_t)kc * TCS_N * 16; };
    for (int bi = 0; bi < nblocks; ++bi) {
        int kc = (std::max(blen[bi], 1) + 3) / 4;
        kc = std::max(2, (kc + 1) & ~1);
        kcs[bi] = kc; boff[bi] = (int64_t)total;
        total += bbytes_of(kc);
    }
    T.blob.assign(total, 0);
    for (int bi = 0; bi < nblocks; ++bi) {
        int8_t* Bm = reinterpret_cast<int8_t*>(T.blob.data() + boff[bi]);
        for (int sidx = 0; sidx < TCS_N; ++sidx) {
            const int slot = bi * TCS_N + sidx;
            const std::vector<int8_t>& c = tab[slot];
            auto at = [&](int ch, int e) -> size_t { return ((size_t)ch * TCS_N + sidx) * 16 + e; };    // byte e of K chunk ch of this slot
            if (c.empty()) {                                       // disabled slot: D = -1 everywhere
                for (int b = 0; b < 4; ++b) Bm[at(0, b)] = -1;
                T.slots[slot].npos = 0;
                continue;
            }
            const int len = (int)c.size() / 4;
            for (int j = 0; j < len; ++j)
                for (int b = 0; b < 4; ++b) Bm[at(j >> 2, 4 * (j & 3) + b)] = c[(size_t)j * 4 + b];
        }
    }
    // Work entries: blocks sorted by length are paired with their neighbour while both B operands fit in shared memory.  Each block
    // of a pair owns one accumulator, so an accumulator is drained (>= ~1000 clocks: TMEM read bandwidth + barrier latencies) under the
    // MMAs of the other block: two long blocks hide each other's drains completely and run at the MMA rate; two short blocks are
    // drain-bound whatever their partner is, so they are best spent on each other.  Initial cost in clocks per tile; scan_impl
    // replaces it with measured clocks after the first batch.
    std::vector<int> ord(nblocks);
    for (int bi = 0; bi < nblocks; ++bi) ord[bi] = bi;
    std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return kcs[x] > kcs[y]; });
    const double drain = 1000.0;
    const size_t b_budget = (size_t)200 * 1024 - (size_t)TCS_STAGES * TCS_STAGE_BYTES;
    std::vector<double> cost;
    for (int i = 0; i < nblocks;) {
        TcBlock e; memset(&e, 0, sizeof e);
        const int L = ord[i];
        e.b_off[0] = boff[L]; e.kchunks[0] = kcs[L]; e.slot0[0] = L * TCS_N; e.nsub = 1;
        size_t bbytes = bbytes_of(kcs[L]);
        if (i + 1 < nblocks && bbytes + bbytes_of(kcs[ord[i + 1]]) <= b_budget) {
            const int S = ord[i + 1];
            e.b_off[1] = boff[S]; e.kchunks[1] = kcs[S]; e.slot0[1] = S * TCS_N; e.nsub = 2;
            bbytes += bbytes_of(kcs[S]);
            // per tile of 512 positions: 4 phases x kchunks / 2 MMAs of 128 clocks each per block; measured on config 4
            // (profiles/r01_scan_tc_role_clocks.txt): 1.19 x the MMA clocks when the MMAs bind, ~8 drains of ~1150 clocks when they do not
            cost.push_back(std::max(1.19 * 4.0 * (kcs[L] + kcs[S]) * 64.0, 8.0 * drain + 1400.0));
            i += 2;
        } else {
            cost.push_back(std::max(1.19 * 4.0 * kcs[L] * 64.0, 4.0 * drain + 700.0));
            i += 1;
        }
        // Tried and removed (git history: 59d1900, 004a558, 1f9ca7b; DESIGN.md 3.1b): four 128-column accumulators for short entries (25 %
        // slower), skipping an all-padding upper column half (slower on config 5), B staged with the 128-byte swizzle (5 % slower).  The
        // generic code paths they needed cost the production kernel 13 % (the MMA warp's instruction stream paces the tensor pipe).
        T.max_b_bytes = std::max(T.max_b_bytes, bbytes);
        T.blocks.push_back(e);
    }
    T.cost = cost;
    return tc_assign_ctas(T.blocks, cost, grid);
}

static int build_plan(mb200_ctx* ctx, const uint16_t* pwms, const int64_t* lens, int K, int maxlen, const uint16_t* thresh,
                      uint32_t flags, int64_t Lb, size_t table_budget, ScanPlan& P) {
    P.K = K;
    std::vector<int> order(K);
    for (int k = 0; k < K; ++k) {
        if (lens[k] < 1 || lens[k] > maxlen)
            MB_FAIL(ctx, MB200_E_INVALID, "motif %d: length %lld outside [1, maxlen=%d]", k, (long long)lens[k], maxlen);
        order[k] = k;
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lens[a] < lens[b]; });
    P.minlen = (int)lens[order[0]];
    P.ngroups = (K + GROUP_MOTIFS - 1) / GROUP_MOTIFS;
    P.K2pad = P.ngroups * GROUP_SLOTS;
    P.pair2motif.assign(P.K2pad / 2, -1);
    P.pairlen.assign(P.K2pad / 2, 0);
    P.em.resize(K);
    auto pw = [&](int k, int a, int ind) -> uint16_t { return pwms[(size_t)k + (size_t)K * ((size_t)a + 4 * (size_t)ind)]; };

    // group lengths, then greedy partition into motif blocks under the shared-memory budget
    std::vector<int> glen(P.ngroups);
    for (int g = 0; g < P.ngroups; ++g) glen[g] = ((int)lens[order[std::min(K - 1, g * GROUP_MOTIFS + GROUP_MOTIFS - 1)]] + 1) & ~1;   // even: zero pad column
    // groups longer than the register-resident fast path (MB200_MAX_MOTIF_LEN columns) go to scan_long_kernel
    int g_long = P.ngroups;
    for (int gq = 0; gq < P.ngroups; ++gq) if (glen[gq] > MB200_MAX_MOTIF_LEN) { g_long = gq; break; }
    int g = 0;
    while (g < g_long) {
        MBlock mb; memset(&mb, 0, sizeof mb);
        mb.g0 = g; size_t tb = 0; int cost = 0;
        while (g < g_long) {
            size_t add = (size_t)glen[g] * COL_BYTES;
            size_t metas = (size_t)(g - mb.g0 + 1) * sizeof(GroupMeta);
            if (g > mb.g0 && tb + add + metas > table_budget) break;
            tb += add; cost += glen[g]; ++g;
        }
        mb.ng = g - mb.g0; mb.tab_bytes = (int32_t)tb; mb.cost = cost;
        mb.blob_bytes = (int32_t)((tb + (size_t)mb.ng * sizeof(GroupMeta) + 15) & ~(size_t)15);
        if ((size_t)mb.blob_bytes > table_budget + 4096)
            MB_FAIL(ctx, MB200_E_UNSUPPORTED, "a single motif group needs %d B of shared memory", mb.blob_bytes);
        P.mblocks.push_back(mb);
    }
    for (int gl = g_long; gl < P.ngroups; ++gl) {
        MBlock mb; memset(&mb, 0, sizeof mb);
        mb.g0 = gl; mb.ng = 1; mb.tab_bytes = glen[gl] * COL_BYTES; mb.cost = glen[gl];
        mb.blob_bytes = (int32_t)(((size_t)mb.tab_bytes + sizeof(GroupMeta) + 15) & ~(size_t)15);
        P.lblocks.push_back(mb);
    }
    size_t total = 0;
    for (auto& mb : P.mblocks) { mb.blob_off = (int64_t)total; total += ((size_t)mb.blob_bytes + 127) & ~(size_t)127; P.max_blob_bytes = std::max(P.max_blob_bytes, mb.blob_bytes); }
    for (auto& mb : P.lblocks) { mb.blob_off = (int64_t)total; total += ((size_t)mb.blob_bytes + 127) & ~(size_t)127; }
    P.blob.assign(total, 0);

    std::vector<MBlock*> all_blocks;
    for (auto& mb : P.mblocks) all_blocks.push_back(&mb);
    for (auto& mb : P.lblocks) all_blocks.push_back(&mb);
    for (MBlock* mbp : all_blocks) {
        MBlock& mb = *mbp;
        uint8_t* tabs = P.blob.data() + mb.blob_off;
        GroupMeta* metas = reinterpret_cast<GroupMeta*>(tabs + mb.tab_bytes);
        int toff = 0;
        for (int gi = 0; gi < mb.ng; ++gi) {
            const int gg = mb.g0 + gi;
            GroupMeta gm; memset(&gm, 0, sizeof gm);
            gm.len = glen[gg]; gm.tab_off = toff;
            uint16_t* T = reinterpret_cast<uint16_t*>(tabs + toff);   // [col][slot][base]
            for (int i = 0; i < GROUP_MOTIFS; ++i) {
                const int idx = gg * GROUP_MOTIFS + i;
                uint16_t thr_f = 0x7C00u, thr_r = 0x7C00u;            // +Inf: never a hit
                if (idx < K) {
                    const int k = order[idx];
                    const int len = (int)lens[k];
                    gm.npos[i] = (int32_t)std::max<int64_t>(0, Lb - len + 1);
                    gm.npos_max = std::max(gm.npos_max, gm.npos[i]);
                    const uint16_t t = hit_threshold(thresh, k);
                    if (flags & MB200_SCAN_FWD) thr_f = t;
                    if (flags & MB200_SCAN_RC) thr_r = t;
                    P.pair2motif[gg * GROUP_MOTIFS + i] = k;
                    P.pairlen[gg * GROUP_MOTIFS + i] = len;
                    P.em[k].slot = gg * GROUP_SLOTS + i * 2;
                    P.em[k].len = len;
                    // table layout [col][slot][base]
                    P.em[k].tab_off = mb.blob_off + toff + (int64_t)i * 16;
                    P.em[k].col_stride = COL_BYTES; P.em[k].base_stride = 2; P.em[k].strand_stride = 8;
                    auto pwk = [&](int a, int ind) { return pw(k, a, ind); };
                    for (int j = 0; j < len; ++j)
                        for (int b = 0; b < 4; ++b) {
                            T[((size_t)j * GROUP_SLOTS + i * 2 + 0) * 4 + b] = mb_eff_entry(pwk, len, b, j, 0);
                            T[((size_t)j * GROUP_SLOTS + i * 2 + 1) * 4 + b] = mb_eff_entry(pwk, len, b, j, 1);
                        }
                }
                gm.thr[i * 2 + 0] = thr_f; gm.thr[i * 2 + 1] = thr_r;
            }
            metas[gi] = gm;
            toff += glen[gg] * COL_BYTES;
        }
    }
    return MB200_OK;
}

// ---- the scan driver: scan_impl runs the stages below; ScanCall holds what they share ----------------------------------------

// What a scan call returns.  Each extern "C" entry point fills one kind; every choice that depends on the mode is made from it.
struct ScanOut {
    enum Kind { HITS, HIST, BEST, SPACING };
    Kind kind = HITS;
    mb200_hit* hits = nullptr; int64_t hits_cap = 0; int64_t* n_hits = nullptr; int64_t* counts = nullptr;   // HITS: as the flags ask
    uint32_t* hist = nullptr;              // HIST: K x HIST_BINS
    mb200_best* best = nullptr;            // BEST: N x K records
    const SpacingJob* sp = nullptr;        // SPACING
};

// Appends n bytes (zeros without src) to a host staging image, padded to `align`; returns their offset.
static size_t put(std::vector<uint8_t>& h, const void* src, size_t n, size_t align = 256) {
    const size_t off = h.size();
    h.resize(off + (n + align - 1) / align * align, 0);
    if (src && n) memcpy(h.data() + off, src, n);
    return off;
}

static const unsigned long long TC_CAP = (unsigned long long)24 << 20;     // candidate records per batch and buffer set
static const int32_t TILE_CHUNKS = 16 * 26;                                  // scan_kernel: position blocks per tile

struct ScanCall {
    mb200_ctx* ctx; const mb200_seqs* seqs; const ScanOut out; const int K; const uint32_t flags;
    const bool keys = out.kind == ScanOut::BEST || out.kind == ScanOut::SPACING;     // best keys and best_reduce_kernel, no hit masks
    const bool want_hits = out.kind == ScanOut::HITS && (flags & MB200_SCAN_WANT_HITS);
    const bool want_counts = out.kind == ScanOut::HITS && (flags & MB200_SCAN_WANT_COUNTS);
    const bool reduce = (flags & MB200_SCAN_REDUCE) && ctx->world > 1;                 // sum the totals across ranks
    int64_t N = 0, Lb = 0, rowwords = 0;
    int grid = 0;
    ScanPlan P;
    TcPlan TP;
    bool use_tc = false;                   // this and later batches take the tensor-core pre-filter + exact verification (scan_tc.cuh)
    bool tc_units = false;                 // the verifier lists the (sequence, motif) units that received a hit
    int32_t W = 0, W16 = 0;                // 32-position mask words and 16-position blocks per sequence
    size_t mask_bytes_per_seq = 0;
    int64_t seqs_per_batch = 0;
    uint32_t* d_mask = nullptr;
    std::vector<uint8_t> h_plan;           // BUF_PLAN's host copy, alive until the final synchronise
    const uint8_t* d_blob = nullptr; const MBlock* d_mblocks = nullptr; const MBlock* d_lblocks = nullptr;
    const int32_t* d_p2m = nullptr; const int32_t* d_plen = nullptr; const EmitMotif* d_em = nullptr;
    int64_t* d_rng = nullptr; unsigned long long* d_counts = nullptr; unsigned long long* d_total = nullptr;
    void (*scan_fn)(const ScanArgs) = nullptr;                     // scan_kernel<RAGGED, BEST> of this call
    int32_t tile_cap_words = 0, blob_cap = 0; size_t smem_bytes = 0;
    int64_t last_nchunks = -1;
    // tensor-core path; counters: [0] reserved, [1] overflow, [2] candidates, [3] hits, [4] listed units, [8 + 2c] clocks and
    // [9 + 2c] tiles of CTA c
    uint8_t* d_tc = nullptr; const TcSlot* d_tc_slots = nullptr; size_t tc_smem = 0, tc_set_stride = 0, tc_uset_stride = 0;
    unsigned long long* d_tc_list = nullptr; unsigned long long* d_tc_ctr = nullptr; uint32_t* d_tc_ulist = nullptr; uint32_t* d_tc_ubits = nullptr;
    unsigned long long tc_stat_cand = 0, tc_stat_hits = 0;
    double tc_stat_macs = 0;               // int8 multiply-adds the tensor core was given (every slot block over every position)
    uint32_t* d_unit_cnt = nullptr; unsigned long long* d_unit_off = nullptr; unsigned long long* d_bsum = nullptr;   // hit lists
    int64_t hits_written = 0, hits_needed = 0;
    unsigned int* d_hist = nullptr;                                                                                   // HIST
    unsigned long long* d_best64 = nullptr; mb200_best* d_best = nullptr; int32_t best_nch = 0;                       // BEST, SPACING
    unsigned int* d_sphist = nullptr; const size_t sphist_bytes = out.sp ? (size_t)out.sp->n_primary * K * 4 * (size_t)out.sp->margin * 4 : 0;   // SPACING
    const mb200_anchor* d_anchors = nullptr; const uint16_t* d_spthr = nullptr; const int32_t* d_mlen = nullptr;
    size_t next_ready = 0;                 // chunks of a pending asynchronous upload this call has waited for
    MbTimers tm{ctx}; int t_total = -1;
    size_t tc_nctr() const { return 8 + 2 * (size_t)grid; }
    size_t tc_ubits_bytes(int64_t ns) const { return (((size_t)ns * (size_t)(P.K2pad / 2) + 31) / 32) * 4; }
};

static int scan_validate(ScanCall& S, const uint16_t* pwms, const int64_t* lens, int maxlen) {
    mb200_ctx* ctx = S.ctx; const ScanOut& o = S.out;
    if (!S.seqs || !pwms || !lens || S.K <= 0 || S.K > 65535 || maxlen <= 0)
        MB_FAIL(ctx, MB200_E_INVALID, "scan: bad arguments (K=%d maxlen=%d)", S.K, maxlen);
    if (!(S.flags & (MB200_SCAN_FWD | MB200_SCAN_RC))) MB_FAIL(ctx, MB200_E_INVALID, "scan: neither FWD nor RC requested");
    if (S.want_hits && (!o.n_hits || (o.hits_cap > 0 && !o.hits))) MB_FAIL(ctx, MB200_E_INVALID, "scan: WANT_HITS needs hits/n_hits");
    if (S.want_counts && !o.counts) MB_FAIL(ctx, MB200_E_INVALID, "scan: WANT_COUNTS needs counts");
    if (S.seqs->device != ctx->device) MB_FAIL(ctx, MB200_E_INVALID, "scan: sequences live on device %d, ctx on %d", S.seqs->device, ctx->device);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    mb_reset_timing(ctx);
    if (o.n_hits) *o.n_hits = 0;
    ctx->held_hits.clear(); ctx->held_hits.shrink_to_fit();
    if (o.counts) memset(o.counts, 0, sizeof(int64_t) * 4 * (size_t)S.K);
    if (o.hist) memset(o.hist, 0, (size_t)S.K * HIST_BINS * 4);
    return MB200_OK;
}

static int scan_plan(ScanCall& S, const uint16_t* pwms, const int64_t* lens, int maxlen, const uint16_t* thresh) {
    mb200_ctx* ctx = S.ctx;
    S.N = S.seqs->N; S.Lb = S.seqs->Lb; S.rowwords = S.seqs->rowwords; S.grid = ctx->sm_count;
    int rc = build_plan(ctx, pwms, lens, S.K, maxlen, thresh, S.flags, S.Lb, 160 * 1024, S.P);
    if (rc) return rc;
    // Thresholded hit lists and counts take the tensor-core path unless the caller or the inputs rule it out; the hit masks, and
    // everything derived from them, are identical either way.
    S.use_tc = S.out.kind == ScanOut::HITS && !(S.flags & MB200_SCAN_NO_TENSOR) && S.Lb < (1ll << 31) &&
               build_tc_plan(S.P, pwms, lens, S.K, thresh, S.flags, S.Lb, S.grid, S.TP);
    ctx->last_scan_path = 0;
    if (S.use_tc) {
        // start from the clocks per tile measured by the previous scan of this ctx when it had the same block structure
        std::vector<int32_t> sig;
        for (auto& e : S.TP.blocks) { sig.push_back(e.nsub); sig.push_back(e.kchunks[0]); sig.push_back(e.kchunks[1]); }
        if (sig == ctx->tc_cost_sig && ctx->tc_cost.size() == S.TP.blocks.size()) { S.TP.cost = ctx->tc_cost; tc_assign_ctas(S.TP.blocks, S.TP.cost, S.grid); }
        else { ctx->tc_cost_sig = sig; ctx->tc_cost.clear(); }
    }
    return MB200_OK;
}

// The totals of a call, K x 4 uint64 counts (WANT_COUNTS) or the K x HIST_BINS uint32 score histogram (HIST), never both: summed
// across ranks (one all-reduce per scan, SURVEY §8e) and copied to the caller.  tm == nullptr: the copy is not timed.
static size_t totals_bytes(const ScanCall& S) { return S.out.hist ? (size_t)S.K * HIST_BINS * 4 : S.want_counts ? (size_t)S.K * 4 * 8 : 0; }
static int copy_totals(ScanCall& S, void* d_totals, MbTimers* tm) {
    mb200_ctx* ctx = S.ctx;
    const size_t bytes = totals_bytes(S);
    if (!bytes) return MB200_OK;
    if (S.reduce) {
        const int rc = S.out.hist ? mb_comm_allreduce_u32(ctx, (unsigned int*)d_totals, bytes / 4) : mb_comm_allreduce_u64(ctx, (unsigned long long*)d_totals, bytes / 8);
        if (rc) return rc;
    }
    const int t = tm ? tm->begin(T_D2H) : -1;
    MB_CUDA(ctx, cudaMemcpyAsync(S.out.hist ? (void*)S.out.hist : (void*)S.out.counts, d_totals, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (tm) tm->end(t);
    return MB200_OK;
}

// Nothing can be scored on this rank (no rows, or no PWM fits a row).  It writes its "none" outputs and still takes part in the
// reduction, with zeroed scratch in place of the counts and the histogram.
static int scan_empty(ScanCall& S) {
    mb200_ctx* ctx = S.ctx; const ScanOut& o = S.out;
    const mb200_best none = {0xFFFFFFFFu, 0, 0, 0};
    if (o.best) std::fill(o.best, o.best + (size_t)S.N * S.K, none);     // no row holds a window (otherwise every batch writes all its records)
    if (o.sp) {                                                          // every secondary is longer than the margin
        memset(o.sp->hist, 0, S.sphist_bytes);
        if (o.sp->sites) std::fill(o.sp->sites, o.sp->sites + (size_t)o.sp->n * S.K, none);
    }
    if (S.reduce && totals_bytes(S)) {
        int rc = mb_ensure_scratch(ctx, totals_bytes(S)); if (rc) return rc;
        MB_CUDA(ctx, cudaMemsetAsync(ctx->scratch, 0, totals_bytes(S), ctx->stream));
        rc = copy_totals(S, ctx->scratch, nullptr); if (rc) return rc;
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return MB200_OK;
}

// BUF_PLAN and the batch size: the masks of a batch stay under 8 GB.
static int stage_plan(ScanCall& S) {
    mb200_ctx* ctx = S.ctx; const ScanPlan& P = S.P;
    const int64_t W64 = (S.Lb - P.minlen + 1 + 31) / 32;
    if (W64 > 0x1fffffff) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "sequence too long");
    S.W = (int32_t)W64; S.W16 = 2 * S.W;
    S.tc_units = S.W <= 4096;
    const size_t off_blob = put(S.h_plan, P.blob.data(), P.blob.size());
    const size_t off_mb = put(S.h_plan, P.mblocks.data(), P.mblocks.size() * sizeof(MBlock));
    const size_t off_lb = put(S.h_plan, P.lblocks.data(), P.lblocks.size() * sizeof(MBlock));
    const size_t off_p2m = put(S.h_plan, P.pair2motif.data(), P.pair2motif.size() * 4);
    const size_t off_plen = put(S.h_plan, P.pairlen.data(), P.pairlen.size() * 4);
    const size_t off_em = put(S.h_plan, P.em.data(), P.em.size() * sizeof(EmitMotif));
    const size_t off_rng = put(S.h_plan, nullptr, (size_t)(S.grid + 1) * 8);
    const size_t off_cnt = put(S.h_plan, nullptr, (size_t)S.K * 4 * 8);
    const size_t off_tot = put(S.h_plan, nullptr, 8);
    int rc = mb_ensure_buf(ctx, BUF_PLAN, S.h_plan.size()); if (rc) return rc;
    uint8_t* d_plan = (uint8_t*)ctx->bufs[BUF_PLAN];
    S.d_blob = d_plan + off_blob; S.d_mblocks = (const MBlock*)(d_plan + off_mb); S.d_lblocks = (const MBlock*)(d_plan + off_lb);
    S.d_p2m = (const int32_t*)(d_plan + off_p2m); S.d_plen = (const int32_t*)(d_plan + off_plen); S.d_em = (const EmitMotif*)(d_plan + off_em);
    S.d_rng = (int64_t*)(d_plan + off_rng); S.d_counts = (unsigned long long*)(d_plan + off_cnt); S.d_total = (unsigned long long*)(d_plan + off_tot);

    const size_t mask_budget = (size_t)8 << 30;
    S.mask_bytes_per_seq = (size_t)S.W * P.K2pad * 4 * (S.keys ? 2 : 1);        // best keys: one 32-bit key per 16-position block
    int64_t spb = std::max<int64_t>(1, (int64_t)(mask_budget / S.mask_bytes_per_seq));
    if (spb > S.N) spb = S.N;
    if ((double)spb * S.W > 2.0e9) spb = std::max<int64_t>(1, (int64_t)(2.0e9 / S.W));
    if (S.out.kind == ScanOut::SPACING) spb = std::max<int64_t>(2, spb & ~(int64_t)1);   // both margins of an anchor in one batch (N is even)
    if (S.use_tc && (double)spb * (double)S.Lb > 2.0e9) spb = std::max<int64_t>(1, (int64_t)(2.0e9 / (double)S.Lb));   // 32-bit virtual positions
    S.seqs_per_batch = spb;
    return MB200_OK;
}

// Tensor-core buffers; BUF_TC_LIST and BUF_TC_UNITS hold two sets each, which the pipelined loop alternates.
static int stage_tc(ScanCall& S) {
    mb200_ctx* ctx = S.ctx; const TcPlan& TP = S.TP;
    std::vector<uint8_t> h_tc;
    put(h_tc, TP.blob.data(), TP.blob.size());
    put(h_tc, TP.blocks.data(), TP.blocks.size() * sizeof(TcBlock));
    const size_t off_slots = put(h_tc, TP.slots.data(), TP.slots.size() * sizeof(TcSlot), 1);
    int rc = mb_ensure_buf(ctx, BUF_TC_PLAN, h_tc.size()); if (rc) return rc;
    const size_t set_bytes = (((size_t)TC_CAP * 8 + S.tc_nctr() * 8) + 255) & ~(size_t)255;
    rc = mb_ensure_buf(ctx, BUF_TC_LIST, 2 * set_bytes); if (rc) return rc;
    S.d_tc = (uint8_t*)ctx->bufs[BUF_TC_PLAN];
    S.d_tc_slots = (const TcSlot*)(S.d_tc + off_slots);
    S.d_tc_list = (unsigned long long*)ctx->bufs[BUF_TC_LIST];
    S.d_tc_ctr = S.d_tc_list + TC_CAP;
    const size_t ubits_bytes = S.tc_ubits_bytes(S.seqs_per_batch) + 256;
    const size_t uset_bytes = (((size_t)TC_CAP * 4 + ubits_bytes) + 255) & ~(size_t)255;
    rc = mb_ensure_buf(ctx, BUF_TC_UNITS, 2 * uset_bytes); if (rc) return rc;
    S.d_tc_ulist = (uint32_t*)ctx->bufs[BUF_TC_UNITS];
    S.d_tc_ubits = S.d_tc_ulist + TC_CAP;
    S.tc_set_stride = set_bytes; S.tc_uset_stride = uset_bytes;
    MB_CUDA(ctx, cudaMemcpyAsync(S.d_tc, h_tc.data(), h_tc.size(), cudaMemcpyHostToDevice, ctx->stream));
    MB_CUDA(ctx, cudaMemsetAsync(S.d_tc_ctr, 0, S.tc_nctr() * 8, ctx->stream));
    MB_CUDA(ctx, cudaMemsetAsync((uint8_t*)S.d_tc_ctr + S.tc_set_stride, 0, S.tc_nctr() * 8, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));           // h_tc goes out of scope
    // at least half of the shared memory: one CTA per SM (each CTA allocates all 512 TMEM columns)
    S.tc_smem = std::max<size_t>((size_t)TCS_STAGES * TCS_STAGE_BYTES + TP.max_b_bytes, (size_t)120 * 1024);
    if (S.tc_smem > ctx->smem_optin) S.use_tc = false;
    else MB_CUDA(ctx, cudaFuncSetAttribute(k_scan_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.tc_smem));
    return MB200_OK;
}

// The device buffers of the call (BUF_* in common.cuh) and the launch set-up of scan_kernel.
static int stage_buffers(ScanCall& S, const int64_t* lens) {
    mb200_ctx* ctx = S.ctx; const int K = S.K;
    int rc = stage_plan(S); if (rc) return rc;
    if (S.use_tc) { rc = stage_tc(S); if (rc) return rc; }
    const int64_t spb = S.seqs_per_batch;
    rc = mb_ensure_buf(ctx, BUF_MASK, (size_t)spb * S.mask_bytes_per_seq); if (rc) return rc;
    S.d_mask = (uint32_t*)ctx->bufs[BUF_MASK];
    if (S.keys) {                                       // per batch: 64-bit best keys, then the records (spacing: the sites)
        rc = mb_ensure_buf(ctx, BUF_UNITS, (size_t)spb * K * 16); if (rc) return rc;
        S.d_best64 = (unsigned long long*)ctx->bufs[BUF_UNITS];
        S.d_best = (mb200_best*)(S.d_best64 + (size_t)spb * K);
        S.best_nch = (S.W16 + BEST_CHUNK - 1) / BEST_CHUNK;
    }
    if (const SpacingJob* sp = S.out.sp) {
        rc = mb_ensure_buf(ctx, BUF_HIST, S.sphist_bytes); if (rc) return rc;
        S.d_sphist = (unsigned int*)ctx->bufs[BUF_HIST];
        std::vector<uint8_t> h;
        std::vector<uint16_t> thr(K); std::vector<int32_t> mlen(K);
        for (int k = 0; k < K; ++k) { thr[k] = hit_threshold(sp->thresh, k); mlen[k] = (int32_t)lens[k]; }
        put(h, sp->anchors, (size_t)sp->n * sizeof(mb200_anchor));
        const size_t off_thr = put(h, thr.data(), (size_t)K * 2), off_len = put(h, mlen.data(), (size_t)K * 4, 1);
        rc = mb_ensure_buf(ctx, BUF_SPACING, h.size()); if (rc) return rc;
        uint8_t* d = (uint8_t*)ctx->bufs[BUF_SPACING];
        MB_CUDA(ctx, cudaMemcpyAsync(d, h.data(), h.size(), cudaMemcpyHostToDevice, ctx->stream));
        MB_CUDA(ctx, cudaMemsetAsync(S.d_sphist, 0, S.sphist_bytes, ctx->stream));
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));         // h goes out of scope
        S.d_anchors = (const mb200_anchor*)d; S.d_spthr = (const uint16_t*)(d + off_thr); S.d_mlen = (const int32_t*)(d + off_len);
    }
    if (S.want_hits) {
        const int64_t units = spb * K * 2, ps_blocks = (units + PS_TILE - 1) / PS_TILE;
        const size_t off_off = ((size_t)units * 4 + 255) & ~(size_t)255;
        const size_t off_bsum = off_off + (((size_t)units * 8 + 255) & ~(size_t)255);
        rc = mb_ensure_buf(ctx, BUF_UNITS, off_bsum + (size_t)ps_blocks * 8 + 256); if (rc) return rc;
        S.d_unit_cnt = (uint32_t*)ctx->bufs[BUF_UNITS];
        S.d_unit_off = (unsigned long long*)((uint8_t*)ctx->bufs[BUF_UNITS] + off_off);
        S.d_bsum = (unsigned long long*)((uint8_t*)ctx->bufs[BUF_UNITS] + off_bsum);
    }
    // scan_kernel: words spanned by a tile: +1 per block inside a sequence, + (rowwords - W16 + 1) when crossing to the next sequence
    const int64_t crossings = (TILE_CHUNKS - 1) / S.W16 + 1;
    const int64_t gap = std::max<int64_t>(0, S.rowwords - (int64_t)S.W16 + 1);
    S.tile_cap_words = (int32_t)(((int64_t)TILE_CHUNKS + crossings * gap + 6 + 4 + 3) & ~(int64_t)3);
    S.blob_cap = (S.P.max_blob_bytes + 127) & ~127;
    S.smem_bytes = (size_t)S.blob_cap + (size_t)S.tile_cap_words * 8 + 64;
    if (S.smem_bytes > ctx->smem_optin) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "scan needs %zu B shared memory (> %zu)", S.smem_bytes, ctx->smem_optin);
    const bool ragged = S.seqs->lens != nullptr;
    S.scan_fn = S.keys ? (ragged ? scan_kernel<true, true> : scan_kernel<false, true>) : (ragged ? scan_kernel<true> : scan_kernel<false>);
    MB_CUDA(ctx, cudaFuncSetAttribute(S.scan_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.smem_bytes));

    S.t_total = S.tm.begin(T_TOTAL);
    const int th = S.tm.begin(T_H2D);
    MB_CUDA(ctx, cudaMemcpyAsync(ctx->bufs[BUF_PLAN], S.h_plan.data(), S.h_plan.size(), cudaMemcpyHostToDevice, ctx->stream));
    S.tm.end(th);
    if (S.out.hist) {
        rc = mb_ensure_buf(ctx, BUF_HIST, (size_t)K * HIST_BINS * 4); if (rc) return rc;
        S.d_hist = (unsigned int*)ctx->bufs[BUF_HIST];
        MB_CUDA(ctx, cudaMemsetAsync(S.d_hist, 0, (size_t)K * HIST_BINS * 4, ctx->stream));
    }
    return MB200_OK;
}

// A batch may start as soon as the chunks of a pending asynchronous upload that hold rows [0, end) are packed (the kernels read a
// few words past the batch's last row: in bounds, and whatever they hold only reaches positions that are masked out).
static int wait_for_rows(ScanCall& S, int64_t end) {
    const mb200_seqs* seqs = S.seqs;
    if (!seqs->pending) return MB200_OK;
    while (S.next_ready < seqs->ready.size() && (S.next_ready == 0 || seqs->ready_end[S.next_ready - 1] < end)) {
        MB_CUDA(S.ctx, cudaStreamWaitEvent(S.ctx->stream, seqs->ready[S.next_ready], 0));
        ++S.next_ready;
    }
    return MB200_OK;
}

// ---- one k_scan_tc batch, shared by the pipelined and the serial loop ------------------------------------------------------------
// make TCS_PROFILE=1, MB200_SCAN_TC_DEBUG=<batch>: the per-role wait clocks of that batch's CTAs (captured by tc_launch)
static void tc_debug_dump(ScanCall& S, const TcArgs& ta) {
#if TCS_PROFILE
    if (!ta.dbg) return;
    std::vector<long long> h((size_t)S.grid * 8);
    cudaStreamSynchronize(S.ctx->stream);
    cudaMemcpy(h.data(), ta.dbg, (size_t)S.grid * 8 * 8, cudaMemcpyDeviceToHost);
    for (int c = 0; c < S.grid; c += 1)
        fprintf(stderr, "[tcdbg] cta %3d blk %lld tiles %lld | mma total %9lld wait_full %9lld wait_acc %9lld | epi total %9lld wait %9lld | prod wait %9lld\n", c, h[c * 8 + 6], h[c * 8 + 7],
                h[c * 8 + 0], h[c * 8 + 1], h[c * 8 + 2], h[c * 8 + 4], h[c * 8 + 3], h[c * 8 + 5]);
#endif
}

// Zeroes the counters, the unit bitmap when given and the part of the mask buffer that ctx->mask_clean_bytes does not cover (the
// buffer is kept all-zero between tensor-core batches), then launches k_scan_tc on ctx->stream.
static int tc_launch(ScanCall& S, int64_t s0, int64_t ns, unsigned long long* list, unsigned long long* ctr, uint32_t* ubits, TcArgs& ta) {
    mb200_ctx* ctx = S.ctx;
    const size_t need = (size_t)ns * S.mask_bytes_per_seq;
    if (ctx->mask_clean_bytes < need) {
        MB_CUDA(ctx, cudaMemsetAsync(S.d_mask, 0, need, ctx->stream));
        ctx->mask_clean_bytes = need;
    }
    MB_CUDA(ctx, cudaMemsetAsync(ctr, 0, 64, ctx->stream));
    if (ubits) MB_CUDA(ctx, cudaMemsetAsync(ubits, 0, S.tc_ubits_bytes(ns), ctx->stream));
    ta.seqw = S.seqs->words; ta.rowwords = S.rowwords; ta.seq0 = s0; ta.lens = S.seqs->lens;
    ta.Lb = (uint32_t)S.Lb; ta.vtotal = (uint32_t)(ns * S.Lb);
    ta.blob = S.d_tc; ta.nblocks = (int32_t)S.TP.blocks.size();
    memset(ta.blocks, 0, sizeof ta.blocks); memcpy(ta.blocks, S.TP.blocks.data(), S.TP.blocks.size() * sizeof(TcBlock));
    ta.slots = S.d_tc_slots;
    ta.list = list; ta.cap = TC_CAP; ta.gcount = ctr; ta.overflow = (uint32_t*)(ctr + 1);
    ta.ntiles = (int32_t)((ns * S.Lb + TCS_TILE - 1) / TCS_TILE);
    for (const TcBlock& e : S.TP.blocks)
        for (int sub = 0; sub < e.nsub; ++sub) S.tc_stat_macs += (double)ta.ntiles * TCS_TILE * TCS_N * e.kchunks[sub] * 16;
    ta.clocks = (long long*)(ctr + 8);
    ta.dbg = nullptr;
#if TCS_PROFILE
    static long long* d_dbg = nullptr;
    const char* e = getenv("MB200_SCAN_TC_DEBUG");
    if (e && s0 / S.seqs_per_batch == atoi(e)) {
        if (!d_dbg) MB_CUDA(ctx, cudaMalloc(&d_dbg, (size_t)S.grid * 8 * 8));
        MB_CUDA(ctx, cudaMemsetAsync(d_dbg, 0, (size_t)S.grid * 8 * 8, ctx->stream)); ta.dbg = d_dbg;
    }
#endif
    const int t_tc = S.tm.begin(T_SCAN);
    k_scan_tc<<<S.grid, TCS_THREADS, S.tc_smem, ctx->stream>>>(ta);
    S.tm.end(t_tc);
    ctx->launches[T_SCAN] += 1;
    return MB200_OK;
}

// The counters h of a finished batch.  false: its candidate list overflowed (thresholds so permissive that most cells pass).
// Otherwise adds its statistics and re-balances the CTAs over the slot blocks with the clocks per tile it measured (the epilogue's
// share depends on the candidate density of a block, which no static model knows).
static bool tc_read_counters(ScanCall& S, const unsigned long long* h) {
    if (h[1]) return false;
    S.tc_stat_cand += h[2]; S.tc_stat_hits += h[3];
    const std::vector<TcBlock>& blocks = S.TP.blocks;
    std::vector<double> cost(blocks.size(), 0.0);
    for (size_t bi = 0; bi < blocks.size(); ++bi) {
        double clk = 0, tiles = 0;
        for (int c = blocks[bi].cta0; c < blocks[bi].cta0 + blocks[bi].nctas; ++c) { clk += (double)h[8 + 2 * c]; tiles += (double)h[8 + 2 * c + 1]; }
        if (tiles <= 0 || clk <= 0) return true;
        cost[bi] = clk / tiles;
    }
    S.ctx->tc_cost = cost;
    tc_assign_ctas(S.TP.blocks, cost, S.grid);
    return true;
}

// Counts-only scans: the pipelined tensor-core path.  The pre-filter of batch i+1 (ctx->stream) runs while batch i is re-scored and
// counted on ctx->aux_stream with the other buffer set, and the host reads batch i's counters while batch i+1 is already running.
// Leaves in todo the batches still to run: those that overflowed (their count is skipped) and those not launched after that.
static int tc_pipelined(ScanCall& S, std::vector<int64_t>& todo) {
    mb200_ctx* ctx = S.ctx; const int grid = S.grid;
    if (!ctx->aux_stream && cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess) MB_FAIL(ctx, MB200_E_CUDA, "scan: cannot create the auxiliary stream");
    cudaStream_t aux = ctx->aux_stream;
    const size_t nctr = S.tc_nctr();
    int rc = mb_ensure_pinned(ctx, 2 * nctr * 8); if (rc) return rc;
    unsigned long long* h_ctr2 = (unsigned long long*)ctx->pinned;
    struct EvGuard {                                            // the events are destroyed on every way out (error returns included)
        cudaEvent_t tc[2] = {nullptr, nullptr}, aux[2] = {nullptr, nullptr};
        ~EvGuard() { for (int b = 0; b < 2; ++b) { if (tc[b]) cudaEventDestroy(tc[b]); if (aux[b]) cudaEventDestroy(aux[b]); } }
    } evg;
    for (int b = 0; b < 2; ++b) { MB_CUDA(ctx, cudaEventCreateWithFlags(&evg.tc[b], cudaEventDisableTiming)); MB_CUDA(ctx, cudaEventCreateWithFlags(&evg.aux[b], cudaEventDisableTiming)); }
    const int nb = (int)todo.size();
    std::vector<char> launched(nb, 0), failed(nb, 0);
    bool overflowed = false;
    auto process = [&](int j) -> int {
        if (cudaEventSynchronize(evg.aux[j & 1]) != cudaSuccess) return MB200_E_CUDA;
        if (!tc_read_counters(S, h_ctr2 + (size_t)(j & 1) * nctr)) { failed[j] = 1; overflowed = true; }
        return MB200_OK;
    };
    int i = 0;
    for (; i < nb && !overflowed; ++i) {
        const int64_t s0 = todo[i];
        const int64_t ns = std::min(S.seqs_per_batch, S.N - s0);
        rc = wait_for_rows(S, s0 + ns); if (rc) return rc;
        const int b = i & 1;
        unsigned long long* list_b = (unsigned long long*)((uint8_t*)S.d_tc_list + (size_t)b * S.tc_set_stride);
        unsigned long long* ctr_b = list_b + TC_CAP;
        uint32_t* ulist_b = (uint32_t*)((uint8_t*)S.d_tc_ulist + (size_t)b * S.tc_uset_stride);
        uint32_t* ubits_b = ulist_b + TC_CAP;
        TcArgs ta;
        rc = tc_launch(S, s0, ns, list_b, ctr_b, nullptr, ta); if (rc) return rc;
        MB_CUDA(ctx, cudaGetLastError());
        MB_CUDA(ctx, cudaEventRecord(evg.tc[b], ctx->stream));
        MB_CUDA(ctx, cudaStreamWaitEvent(aux, evg.tc[b], 0));
        MB_CUDA(ctx, cudaMemsetAsync(ubits_b, 0, S.tc_ubits_bytes(ns), aux));
        const int t_vf = S.tm.begin_on(T_EMIT, aux);
        // 128-thread blocks: next to a k_scan_tc CTA (608 threads x 96 registers) an SM has ~7 K registers left
        k_scan_tc_verify<<<grid * 16, 128, 0, aux>>>(list_b, ctr_b, TC_CAP, ta.slots, S.d_em, S.d_blob, S.seqs->words, S.rowwords, s0, (uint32_t)S.Lb,
                                                    S.W, S.P.K2pad, S.d_mask, ctr_b + 2, ubits_b, ulist_b, ctr_b + 4, S.seqs->lens);
        S.tm.end_on(t_vf, aux);
        const int t_ct = S.tm.begin_on(T_COUNT, aux);
        count_listed_kernel<<<grid * 16, 128, 0, aux>>>(S.d_mask, ulist_b, ctr_b + 4, S.W, S.P.K2pad, S.d_p2m, S.d_plen, S.d_counts, ctr_b + 1, nullptr, 0, 1);
        S.tm.end_on(t_ct, aux);
        MB_CUDA(ctx, cudaGetLastError());
        MB_CUDA(ctx, cudaMemcpyAsync(h_ctr2 + (size_t)b * nctr, ctr_b, nctr * 8, cudaMemcpyDeviceToHost, aux));
        MB_CUDA(ctx, cudaEventRecord(evg.aux[b], aux));
        ctx->launches[T_EMIT] += 1; ctx->launches[T_COUNT] += 1;
        launched[i] = 1;
        tc_debug_dump(S, ta);
        if (i >= 1) { rc = process(i - 1); if (rc) return rc; }
    }
    // every batch but the last launched one was looked at inside the loop
    if (i > 0) { rc = process(i - 1); if (rc) return rc; }
    MB_CUDA(ctx, cudaStreamSynchronize(aux));
    std::vector<int64_t> rest;
    for (int j = 0; j < nb; ++j) if (!launched[j] || failed[j]) rest.push_back(todo[j]);
    todo.swap(rest);
    if (overflowed) { S.use_tc = false; ctx->last_scan_path = 2; ctx->mask_clean_bytes = 0; }     // a failed batch may have left bits behind (its count was skipped)
    else ctx->last_scan_path = 1;
    return MB200_OK;
}

// A tensor-core batch outside the pipeline: pre-filter and verifier on ctx->stream, and the host reads the counters before the next
// batch.  *done: the masks are complete.  After a candidate-list overflow this and every later batch take scan_kernel.
static int tc_serial_batch(ScanCall& S, int64_t s0, int64_t ns, bool* done) {
    mb200_ctx* ctx = S.ctx;
    TcArgs ta;
    int rc = tc_launch(S, s0, ns, S.d_tc_list, S.d_tc_ctr, S.tc_units ? S.d_tc_ubits : nullptr, ta); if (rc) return rc;
    const int t_vf = S.tm.begin(T_EMIT);
    k_scan_tc_verify<<<S.grid * 8, 256, 0, ctx->stream>>>(S.d_tc_list, S.d_tc_ctr, TC_CAP, ta.slots, S.d_em, S.d_blob, S.seqs->words, S.rowwords, s0,
                                                         (uint32_t)S.Lb, S.W, S.P.K2pad, S.d_mask, S.d_tc_ctr + 2,
                                                         S.tc_units ? S.d_tc_ubits : nullptr, S.d_tc_ulist, S.d_tc_ctr + 4, S.seqs->lens);
    S.tm.end(t_vf);
    ctx->launches[T_EMIT] += 1;
    MB_CUDA(ctx, cudaGetLastError());
    std::vector<unsigned long long> h_ctr(S.tc_nctr(), 0);
    MB_CUDA(ctx, cudaMemcpyAsync(h_ctr.data(), S.d_tc_ctr, h_ctr.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    tc_debug_dump(S, ta);
    *done = tc_read_counters(S, h_ctr.data());
    ctx->mask_clean_bytes = 0;                               // the verifier has set bits (re-established when the listed count or clear_listed_kernel clears them)
    if (!*done) { S.use_tc = false; ctx->last_scan_path = 2; }
    else if (ctx->last_scan_path == 0) ctx->last_scan_path = 1;
    return MB200_OK;
}

// ---- scan_kernel / scan_long_kernel --------------------------------------------------------------------------------------------
// Per-CTA ranges of (motif block, tile) pairs for each new batch shape: a contiguous split, mblock-major, weighted by column count.
static int update_cta_ranges(ScanCall& S, int64_t ns) {
    const int64_t nchunks = ns * (int64_t)S.W16;
    if (nchunks == S.last_nchunks) return MB200_OK;
    const std::vector<MBlock>& mblocks = S.P.mblocks;
    const int grid = S.grid;
    const int64_t ntiles = (nchunks + TILE_CHUNKS - 1) / TILE_CHUNKS;
    std::vector<int64_t> h_rng(grid + 1);
    double total_cost = 0;
    for (auto& mb : mblocks) total_cost += (double)mb.cost * (double)ntiles;
    size_t mbi = 0; double acc = 0; int64_t q = 0;
    h_rng[0] = 0;
    for (int b = 1; b <= grid; ++b) {
        const double target = total_cost * b / grid;
        while (mbi < mblocks.size()) {
            const double c = (double)mblocks[mbi].cost;
            const int64_t qend = (int64_t)(mbi + 1) * ntiles;
            int64_t take = (int64_t)((target - acc) / c + 0.5);
            if (take < 0) take = 0;
            if (q + take >= qend) { acc += (double)(qend - q) * c; q = qend; ++mbi; }
            else { acc += (double)take * c; q += take; break; }
        }
        h_rng[b] = (b == grid) ? (int64_t)mblocks.size() * ntiles : q;
    }
    MB_CUDA(S.ctx, cudaMemcpyAsync(S.d_rng, h_rng.data(), (size_t)(grid + 1) * 8, cudaMemcpyHostToDevice, S.ctx->stream));
    MB_CUDA(S.ctx, cudaStreamSynchronize(S.ctx->stream));   // h_rng goes out of scope
    S.last_nchunks = nchunks;
    return MB200_OK;
}

static void simt_batch(ScanCall& S, int64_t s0, int64_t ns) {
    mb200_ctx* ctx = S.ctx; const ScanPlan& P = S.P;
    const int t1 = S.tm.begin(T_SCAN);
    ctx->mask_clean_bytes = 0;
    if (!P.mblocks.empty()) {
        ScanArgs a;
        a.seqw = S.seqs->words; a.rowwords = S.rowwords; a.W = S.W16;
        a.chunk0 = s0 * (int64_t)S.W16; a.nchunks = ns * (int64_t)S.W16;
        a.mask = S.d_mask; a.K2pad = P.K2pad;
        a.blob = S.d_blob; a.mblocks = S.d_mblocks; a.n_mblocks = (int32_t)P.mblocks.size();
        a.tile_chunks = TILE_CHUNKS; a.ntiles = (a.nchunks + TILE_CHUNKS - 1) / TILE_CHUNKS; a.tile_cap_words = S.tile_cap_words; a.blob_cap_bytes = S.blob_cap;
        a.cta_range = S.d_rng;
        a.lens = S.seqs->lens; a.Lb = S.Lb;
        S.scan_fn<<<S.grid, SCAN_THREADS, S.smem_bytes, ctx->stream>>>(a);
        ctx->launches[T_SCAN] += 1;
    }
    if (!P.lblocks.empty()) {
        const int64_t warps = ns * (int64_t)P.lblocks.size() * GROUP_SLOTS;
        auto long_kernel = S.keys ? scan_long_kernel<true> : scan_long_kernel<false>;
        long_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, ctx->stream>>>(S.seqs->words, S.rowwords, s0, ns, S.W, P.K2pad, S.d_blob,
                                                                               S.d_lblocks, (int32_t)P.lblocks.size(), S.d_mask, S.seqs->lens, S.Lb);
        ctx->launches[T_SCAN] += 1;
    }
    S.tm.end(t1);
}

// ---- per-batch output stages ----------------------------------------------------------------------------------------------------
// Counts from the masks: chromosome-scale rows without a hit list take the blocked count_long_*; after the tensor-core verifier
// only the listed units have hits (counts only: counted and cleared; with a hit list: their counts feed the prefix sum, zero
// elsewhere, and the words stay until emit_kernel has read them); otherwise count_kernel walks every unit.
static int count_batch(ScanCall& S, int64_t ns, bool tc_done) {
    mb200_ctx* ctx = S.ctx; const int32_t W = S.W, K2pad = S.P.K2pad, Pp = K2pad / 2;
    const int t2 = S.tm.begin(T_COUNT);
    if (!S.want_hits && W > 4096) {
        const int32_t WB = 512, nblocks = (W + WB - 1) / WB;
        const int64_t nbt = ns * (int64_t)nblocks * Pp;
        const size_t o_top1 = 0, o_top2 = o_top1 + (size_t)ns * Pp * 8, o_nh = o_top2 + (size_t)ns * Pp * 8, o_dup = o_nh + (size_t)ns * Pp * 4;
        const size_t o_cand = (o_dup + (size_t)ns * Pp * 4 + 255) & ~(size_t)255;
        const int rc = mb_ensure_buf(ctx, BUF_LONG_COUNT, o_cand + (size_t)nbt * sizeof(LongCand)); if (rc) return rc;
        uint8_t* lb = (uint8_t*)ctx->bufs[BUF_LONG_COUNT];
        MB_CUDA(ctx, cudaMemsetAsync(lb, 0, o_cand, ctx->stream));
        count_long_a<<<(unsigned)((nbt + 255) / 256), 256, 0, ctx->stream>>>(S.d_mask, ns, W, K2pad, WB, nblocks, S.d_p2m, S.d_plen, S.d_counts,
            (unsigned long long*)(lb + o_top1), (unsigned int*)(lb + o_nh), (LongCand*)(lb + o_cand));
        count_long_b<<<(unsigned)((nbt + 255) / 256), 256, 0, ctx->stream>>>(ns, Pp, nblocks, (const LongCand*)(lb + o_cand), (const unsigned long long*)(lb + o_top1),
            (unsigned long long*)(lb + o_top2), (unsigned int*)(lb + o_dup));
        count_long_c<<<(unsigned)((ns * Pp + 255) / 256), 256, 0, ctx->stream>>>(ns, Pp, S.d_p2m, S.d_plen,
            (const unsigned long long*)(lb + o_top1), (const unsigned long long*)(lb + o_top2), (const unsigned int*)(lb + o_dup), (const unsigned int*)(lb + o_nh), S.d_counts);
        ctx->launches[T_COUNT] += 3;
    } else if (tc_done && S.tc_units) {
        if (S.want_hits) MB_CUDA(ctx, cudaMemsetAsync(S.d_unit_cnt, 0, (size_t)ns * S.K * 2 * 4, ctx->stream));
        count_listed_kernel<<<S.grid * 8, 256, 0, ctx->stream>>>(S.d_mask, S.d_tc_ulist, S.d_tc_ctr + 4, W, K2pad, S.d_p2m, S.d_plen, S.d_counts, nullptr,
                                                                  S.want_hits ? S.d_unit_cnt : nullptr, S.K, S.want_hits ? 0 : 1);
        ctx->launches[T_COUNT] += 1;
        if (!S.want_hits) ctx->mask_clean_bytes = (size_t)ns * S.mask_bytes_per_seq;   // every word with a bit belongs to a listed unit and was cleared
    } else {
        count_kernel<<<(unsigned)((ns * Pp + 255) / 256), 256, 0, ctx->stream>>>(S.d_mask, ns, W, K2pad, S.d_p2m, S.d_plen, S.d_counts, S.d_unit_cnt, S.K);
        ctx->launches[T_COUNT] += 1;
    }
    S.tm.end(t2);
    MB_CUDA(ctx, cudaGetLastError());
    return MB200_OK;
}

// Hit list of a batch: prefix sum over the unit counts, emit_kernel, copy to the caller's array (or, once it is outgrown, to the
// list held in the ctx), then clear the listed words of the tensor-core path.
static int emit_batch(ScanCall& S, int64_t s0, int64_t ns, bool tc_done) {
    mb200_ctx* ctx = S.ctx; const ScanOut& o = S.out;
    const int64_t units = ns * S.K * 2;
    const int64_t nb = (units + PS_TILE - 1) / PS_TILE;
    const int t3 = S.tm.begin(T_EMIT);
    ps_block_sums<<<(unsigned)nb, PS_THREADS, 0, ctx->stream>>>(S.d_unit_cnt, units, S.d_bsum);
    ps_scan_sums<<<1, PS_THREADS, 0, ctx->stream>>>(S.d_bsum, nb, S.d_total);
    ps_apply<<<(unsigned)nb, PS_THREADS, 0, ctx->stream>>>(S.d_unit_cnt, units, S.d_bsum, S.d_unit_off);
    S.tm.end(t3);
    ctx->launches[T_EMIT] += 3;
    unsigned long long h_total = 0;
    MB_CUDA(ctx, cudaMemcpyAsync(&h_total, S.d_total, 8, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    S.hits_needed += (int64_t)h_total;
    // a list that outgrows the caller's buffer is kept in the ctx (host memory) and handed over by mb200_scan_take_hits:
    // the caller's retry does not pay for the scan, count and prefix kernels a second time
    const bool spill = S.hits_needed > o.hits_cap;
    if (spill && ctx->held_hits.empty() && S.hits_written) ctx->held_hits.assign(o.hits, o.hits + S.hits_written);
    if (h_total) {
        const int rc = mb_ensure_buf(ctx, BUF_HITS, (size_t)h_total * sizeof(mb200_hit)); if (rc) return rc;
        mb200_hit* d_hits = (mb200_hit*)ctx->bufs[BUF_HITS];
        const int t4 = S.tm.begin(T_EMIT);
        emit_kernel<<<(unsigned)((units + 255) / 256), 256, 0, ctx->stream>>>(S.d_mask, S.seqs->words, S.rowwords, s0, ns, S.W, S.P.K2pad, S.K,
                                                                           S.d_em, S.d_blob, S.d_unit_cnt, S.d_unit_off, d_hits);
        S.tm.end(t4);
        ctx->launches[T_EMIT] += 1;
        MB_CUDA(ctx, cudaGetLastError());
        const int t5 = S.tm.begin(T_D2H);
        mb200_hit* dst = o.hits + S.hits_written;
        if (spill) { ctx->held_hits.resize((size_t)S.hits_written + (size_t)h_total); dst = ctx->held_hits.data() + S.hits_written; }
        MB_CUDA(ctx, cudaMemcpyAsync(dst, d_hits, (size_t)h_total * sizeof(mb200_hit), cudaMemcpyDeviceToHost, ctx->stream));
        S.tm.end(t5);
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        S.hits_written += (int64_t)h_total;
    }
    if (tc_done && S.tc_units) {
        clear_listed_kernel<<<S.grid * 8, 256, 0, ctx->stream>>>(S.d_mask, S.d_tc_ulist, S.d_tc_ctr + 4, S.W, S.P.K2pad);
        ctx->launches[T_EMIT] += 1;
        ctx->mask_clean_bytes = (size_t)ns * S.mask_bytes_per_seq;
    }
    return MB200_OK;
}

static int hist_batch(ScanCall& S, int64_t s0, int64_t ns) {
    mb200_ctx* ctx = S.ctx;
    const int64_t units = ns * S.K * 2;
    const int t7 = S.tm.begin(T_EMIT);
    hist_kernel<<<(unsigned)((units + 255) / 256), 256, 0, ctx->stream>>>(S.d_mask, S.seqs->words, S.rowwords, s0, ns, S.W, S.P.K2pad, S.K, S.d_em, S.d_blob, S.d_hist);
    S.tm.end(t7);
    ctx->launches[T_EMIT] += 1;
    MB_CUDA(ctx, cudaGetLastError());
    return MB200_OK;
}

// Best keys of a batch reduced to one 64-bit slot per (row, motif), then records to the caller (BEST) or, for anchors s0/2 ..
// (s0 + ns)/2, counts into the spacing histogram and the sites when asked (SPACING).
static int best_batch(ScanCall& S, int64_t s0, int64_t ns) {
    mb200_ctx* ctx = S.ctx; const SpacingJob* sp = S.out.sp; const int K = S.K;
    const int t2 = S.tm.begin(T_COUNT);
    MB_CUDA(ctx, cudaMemsetAsync(S.d_best64, 0, (size_t)ns * K * 8, ctx->stream));
    const int64_t rthreads = ns * (int64_t)S.best_nch * (S.P.K2pad / 2);
    best_reduce_kernel<<<(unsigned)((rthreads + 255) / 256), 256, 0, ctx->stream>>>(S.d_mask, ns, S.W16, S.P.K2pad, S.best_nch, S.d_p2m, K, S.d_best64);
    mb200_best* dst = nullptr; int64_t n = 0;
    if (sp) {
        const int64_t na = ns / 2;
        spacing_kernel<<<(unsigned)((na * K + 255) / 256), 256, 0, ctx->stream>>>(S.d_best64, na, K, S.d_anchors + s0 / 2, S.d_spthr, S.d_mlen, sp->margin,
                                                                                 S.d_sphist, sp->sites ? S.d_best : nullptr);
        if (sp->sites) { dst = sp->sites + (size_t)(s0 / 2) * K; n = na * K; }
    } else {
        best_finalize_kernel<<<(unsigned)((ns * K + 255) / 256), 256, 0, ctx->stream>>>(S.d_best64, ns * K, S.d_best);
        dst = S.out.best + (size_t)s0 * K; n = ns * K;
    }
    S.tm.end(t2);
    ctx->launches[T_COUNT] += 2;
    MB_CUDA(ctx, cudaGetLastError());
    if (dst) {
        const int t6 = S.tm.begin(T_D2H);
        MB_CUDA(ctx, cudaMemcpyAsync(dst, S.d_best, (size_t)n * sizeof(mb200_best), cudaMemcpyDeviceToHost, ctx->stream));
        S.tm.end(t6);
    }
    return MB200_OK;
}

// One batch outside the pipelined loop: the masks (or best keys), then the output stage of the mode.
static int run_batch(ScanCall& S, int64_t s0, int64_t ns) {
    int rc = wait_for_rows(S, s0 + ns); if (rc) return rc;
    rc = update_cta_ranges(S, ns); if (rc) return rc;
    bool tc_done = false;
    if (S.use_tc) { rc = tc_serial_batch(S, s0, ns, &tc_done); if (rc) return rc; }
    if (!tc_done) simt_batch(S, s0, ns);
    MB_CUDA(S.ctx, cudaGetLastError());
    if (S.keys) return best_batch(S, s0, ns);                       // BEST, SPACING
    rc = count_batch(S, ns, tc_done); if (rc) return rc;            // HITS, HIST
    if (S.out.hist) return hist_batch(S, s0, ns);
    return S.want_hits ? emit_batch(S, s0, ns, tc_done) : MB200_OK;
}

static int scan_finish(ScanCall& S) {
    mb200_ctx* ctx = S.ctx; const ScanOut& o = S.out;
    int rc = copy_totals(S, o.hist ? (void*)S.d_hist : (void*)S.d_counts, &S.tm); if (rc) return rc;
    if (o.sp) {
        const int t9 = S.tm.begin(T_D2H);
        MB_CUDA(ctx, cudaMemcpyAsync(o.sp->hist, S.d_sphist, S.sphist_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        S.tm.end(t9);
    }
    S.tm.end(S.t_total);
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    S.tm.collect();
    if (S.d_tc_ctr && getenv("MB200_SCAN_TC_STATS")) {
        fprintf(stderr, "[mb200] tensor-core scan: %s, candidates %llu, hits %llu, scan %.3f ms, count %.3f ms, int8 MACs %.4e\n", S.use_tc ? "used" : "fell back",
                S.tc_stat_cand, S.tc_stat_hits, ctx->ms[T_SCAN], ctx->ms[T_COUNT], S.tc_stat_macs);
    }
    if (S.seqs->pending) { rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(S.seqs)); if (rc) return rc; }      // the upload has completed: report bad symbols
    if (o.n_hits) *o.n_hits = S.hits_needed;
    if (S.want_hits && S.hits_needed > o.hits_cap)
        MB_FAIL(ctx, MB200_E_HITS_OVERFLOW, "scan: %lld hits, capacity %lld", (long long)S.hits_needed, (long long)o.hits_cap);
    return MB200_OK;
}

static int32_t scan_impl(mb200_ctx* ctx, const mb200_seqs* seqs, const uint16_t* pwms_f16, const int64_t* lens, int32_t K,
                         int32_t maxlen, const uint16_t* thresh_f16, uint32_t flags, const ScanOut& out) {
    if (!ctx) return MB200_E_INVALID;
    ScanCall S{ctx, seqs, out, K, flags};
    int rc = scan_validate(S, pwms_f16, lens, maxlen); if (rc) return rc;
    rc = scan_plan(S, pwms_f16, lens, maxlen, thresh_f16); if (rc) return rc;
    if (S.N == 0 || S.Lb - S.P.minlen + 1 <= 0) return scan_empty(S);
    rc = stage_buffers(S, lens); if (rc) return rc;
    std::vector<int64_t> todo;                                     // first rows of the batches still to run
    for (int64_t s0 = 0; s0 < S.N; s0 += S.seqs_per_batch) todo.push_back(s0);
    if (S.use_tc && !S.want_hits && S.tc_units) { rc = tc_pipelined(S, todo); if (rc) return rc; }
    for (const int64_t s0 : todo) { rc = run_batch(S, s0, std::min(S.seqs_per_batch, S.N - s0)); if (rc) return rc; }
    return scan_finish(S);
}

extern "C" int32_t mb200_scan(mb200_ctx* ctx, const mb200_seqs* seqs, const uint16_t* pwms_f16, const int64_t* lens, int32_t K,
                              int32_t maxlen, const uint16_t* thresh_f16, uint32_t flags, mb200_hit* hits, int64_t hits_cap,
                              int64_t* n_hits, int64_t* counts) {
    ScanOut out; out.hits = hits; out.hits_cap = hits_cap; out.n_hits = n_hits; out.counts = counts;
    return scan_impl(ctx, seqs, pwms_f16, lens, K, maxlen, thresh_f16, flags, out);
}

// Diagnostic (host arithmetic only, ctx-free): the tensor-core pre-filter's error bound and threshold for one (motif, strand) slot.
// cols_f16: len x 4 Float16 bit patterns, row = PWM column in scoring order, entries {A,C,G,T}; thresh_f16 as passed to mb200_scan.
extern "C" int32_t mb200_scan_prefilter_bound(const uint16_t* cols_f16, int32_t len, uint16_t thresh_f16, double* E, double* t_prefilter,
                                              uint16_t* col0_f16, int32_t* possible) {
    if (!cols_f16 || len < 1 || len > MB200_MAX_MOTIF_LEN || !E || !t_prefilter || !possible) return MB200_E_INVALID;
    std::vector<double> w((size_t)len * 4);
    double A = 0.0;
    for (int j = 0; j < len; ++j) {
        double am = 0.0;
        for (int b = 0; b < 4; ++b) {
            if (h16_nonfinite(cols_f16[j * 4 + b])) return MB200_E_UNSUPPORTED;
            w[(size_t)j * 4 + b] = (double)h16_to_float(cols_f16[j * 4 + b]);
            am = std::max(am, std::fabs(w[(size_t)j * 4 + b]));
        }
        A += am;
    }
    if (h16_nonfinite(thresh_f16)) return MB200_E_UNSUPPORTED;
    const double t = std::max(0.0, (double)h16_to_float(thresh_f16));
    *E = 0.0; *t_prefilter = 0.0;
    *possible = tc_prefilter_threshold(w, len, t, A, E, t_prefilter) ? 1 : 0;
    if (*possible && col0_f16) for (int b = 0; b < 4; ++b) col0_f16[b] = h16_round_up(w[b] - *t_prefilter);      // what column 0 of the B operand holds
    return MB200_OK;
}

// Diagnostic (host arithmetic only, ctx-free): the int8 B operand of one slot, as k_scan_tc multiplies it.  Same arguments as
// mb200_scan_prefilter_bound; e: the scale 2^e, k: the len column offsets, q: len x 4 entries (tc_int8_filter).
extern "C" int32_t mb200_scan_prefilter_int8(const uint16_t* cols_f16, int32_t len, uint16_t thresh_f16, int32_t* e, int32_t* k, int8_t* q,
                                             int32_t* possible) {
    if (!e || !k || !q) return MB200_E_INVALID;
    double E = 0.0, tp = 0.0;
    uint16_t col0[4];
    const int32_t rc = mb200_scan_prefilter_bound(cols_f16, len, thresh_f16, &E, &tp, col0, possible);
    if (rc || !*possible) return rc;
    std::vector<double> f((size_t)len * 4);
    for (int j = 0; j < len; ++j)
        for (int b = 0; b < 4; ++b) f[(size_t)j * 4 + b] = (double)h16_to_float(j ? cols_f16[j * 4 + b] : col0[b]);
    *e = tc_int8_filter(f, len, q, k);
    return MB200_OK;
}

// the complete hit list of the last mb200_scan of this ctx that returned MB200_E_HITS_OVERFLOW (kept on the host by the library)
extern "C" int32_t mb200_scan_take_hits(mb200_ctx* ctx, mb200_hit* hits, int64_t hits_cap, int64_t* n_hits) {
    if (!ctx || !n_hits) return MB200_E_INVALID;
    *n_hits = (int64_t)ctx->held_hits.size();
    if (*n_hits == 0) MB_FAIL(ctx, MB200_E_INVALID, "scan_take_hits: no overflowed hit list is held");
    if (hits_cap < *n_hits || !hits) MB_FAIL(ctx, MB200_E_HITS_OVERFLOW, "scan_take_hits: %lld hits, capacity %lld", (long long)*n_hits, (long long)hits_cap);
    memcpy(hits, ctx->held_hits.data(), (size_t)*n_hits * sizeof(mb200_hit));
    ctx->held_hits.clear(); ctx->held_hits.shrink_to_fit();
    return MB200_OK;
}

extern "C" int32_t mb200_scan_last_path(const mb200_ctx* ctx) { return ctx ? ctx->last_scan_path : MB200_E_INVALID; }

// hist: K * 32768 uint32, hist[k][b] = number of hits (score > 0, both requested strands) whose Float16 score has bit pattern b.
extern "C" int32_t mb200_scan_hist(mb200_ctx* ctx, const mb200_seqs* seqs, const uint16_t* pwms_f16, const int64_t* lens, int32_t K,
                                   int32_t maxlen, uint32_t flags, uint32_t* hist) {
    if (!ctx) return MB200_E_INVALID;
    if (!hist) MB_FAIL(ctx, MB200_E_INVALID, "scan_hist: null histogram");
    const uint32_t f = (flags & (MB200_SCAN_FWD | MB200_SCAN_RC | MB200_SCAN_REDUCE));
    ScanOut out; out.kind = ScanOut::HIST; out.hist = hist;
    return scan_impl(ctx, seqs, pwms_f16, lens, K, maxlen, nullptr, f, out);
}

extern "C" int32_t mb200_scan_best(mb200_ctx* ctx, const mb200_seqs* seqs, const uint16_t* pwms_f16, const int64_t* lens, int32_t K,
                                   int32_t maxlen, uint32_t flags, mb200_best* best) {
    if (!ctx) return MB200_E_INVALID;
    if (!best) MB_FAIL(ctx, MB200_E_INVALID, "scan_best: null output");
    if (flags & ~(MB200_SCAN_FWD | MB200_SCAN_RC)) MB_FAIL(ctx, MB200_E_INVALID, "scan_best: flags 0x%x: only MB200_SCAN_FWD | MB200_SCAN_RC", flags);
    ScanOut out; out.kind = ScanOut::BEST; out.best = best;
    return scan_impl(ctx, seqs, pwms_f16, lens, K, maxlen, nullptr, flags, out);
}

// The margins of every anchor become rows 2i (left) and 2i + 1 (right) of a fixed-length store (mb200_seqs_windows); the best-site
// scan of that store feeds spacing_kernel batch by batch, and only the histogram (and the sites, when asked) comes back.
extern "C" int32_t mb200_scan_spacing(mb200_ctx* ctx, const mb200_seqs* seqs, const mb200_anchor* anchors, int64_t n_anchors,
                                      int32_t n_primary, int32_t margin, const uint16_t* pwms_f16, const int64_t* lens, int32_t K,
                                      int32_t maxlen, const uint16_t* thresh_f16, uint32_t* hist, mb200_best* sites) {
    if (!ctx) return MB200_E_INVALID;
    if (!seqs || !hist || !pwms_f16 || !lens || K <= 0 || K > 65535 || n_anchors < 0 || (n_anchors > 0 && !anchors))
        MB_FAIL(ctx, MB200_E_INVALID, "scan_spacing: bad arguments (K=%d n_anchors=%lld)", K, (long long)n_anchors);
    if (margin < 1 || margin > 65536) MB_FAIL(ctx, MB200_E_INVALID, "scan_spacing: margin %d outside [1, 65536]", margin);
    if (n_primary < 1 || n_primary > 65535) MB_FAIL(ctx, MB200_E_INVALID, "scan_spacing: n_primary %d outside [1, 65535]", n_primary);
    std::vector<int64_t> row((size_t)n_anchors * 2), start((size_t)n_anchors * 2);
    for (int64_t i = 0; i < n_anchors; ++i) {
        const mb200_anchor& a = anchors[i];
        if (a.primary >= n_primary || a.comp > 1 || a.len < 1 || a.row < 0 || a.row >= seqs->N)
            MB_FAIL(ctx, MB200_E_INVALID, "scan_spacing: anchor %lld: primary %d comp %d len %d row %lld", (long long)i, (int)a.primary, (int)a.comp, a.len, (long long)a.row);
        if (a.start - margin < 0 || a.start > mb_row_len(seqs, a.row) - a.len - margin)
            MB_FAIL(ctx, MB200_E_INVALID, "scan_spacing: anchor %lld: flank [%lld, %lld) leaves row %lld (%lld bases)", (long long)i, (long long)(a.start - margin),
                    (long long)(a.start + a.len + margin), (long long)a.row, (long long)mb_row_len(seqs, a.row));
        row[2 * i] = row[2 * i + 1] = a.row;
        start[2 * i] = a.start - margin;
        start[2 * i + 1] = a.start + a.len;
    }
    if (n_anchors == 0) { mb_reset_timing(ctx); memset(hist, 0, (size_t)n_primary * K * 4 * (size_t)margin * 4); return MB200_OK; }
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    struct Guard {                                      // events and the margin store are released on every way out (error returns included)
        mb200_ctx* ctx; cudaEvent_t e0 = nullptr, e1 = nullptr; mb200_seqs* win = nullptr;
        ~Guard() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); if (win) mb200_seqs_free(ctx, win); }
    } g{ctx};
    MB_CUDA(ctx, cudaEventCreate(&g.e0));
    MB_CUDA(ctx, cudaEventCreate(&g.e1));
    MB_CUDA(ctx, cudaEventRecord(g.e0, ctx->stream));
    int rc = mb200_seqs_windows(ctx, seqs, row.data(), start.data(), 2 * n_anchors, margin, &g.win);
    if (rc) return rc;
    MB_CUDA(ctx, cudaEventRecord(g.e1, ctx->stream));
    MB_CUDA(ctx, cudaEventSynchronize(g.e1));
    float pack_ms = 0;
    MB_CUDA(ctx, cudaEventElapsedTime(&pack_ms, g.e0, g.e1));
    const SpacingJob job = {anchors, n_anchors, n_primary, margin, thresh_f16, hist, sites};
    ScanOut out; out.kind = ScanOut::SPACING; out.sp = &job;
    rc = scan_impl(ctx, g.win, pwms_f16, lens, K, maxlen, nullptr, MB200_SCAN_FWD | MB200_SCAN_RC, out);
    if (rc) return rc;
    ctx->ms[T_PACK] += pack_ms; ctx->ms[T_TOTAL] += pack_ms; ctx->launches[T_PACK] += 1;       // scan_impl reset the timing
    return MB200_OK;
}
