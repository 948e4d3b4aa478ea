// Tensor-core pre-filter for the thresholded PWM scan (tcgen05.mma kind::i8, exact int32 accumulators in TMEM) + exact verification.
//
// What it replaces: the same reference functions as scan_kernel (greedy_search! _h3_1_alignment.jl:18-36 followed by
// filter_position_by_best_thresh! _s2_filter_pos_w_scores.jl:116-125), for the case the fused-threshold callers use
// (thresh given).  The reference's score is a LEFT-TO-RIGHT Float16 running sum; a GEMM cannot reproduce its rounding, so the
// GEMM is only a FILTER and every position it lets through is re-scored with the sequential Float16 adds:
//
//   1. k_scan_tc: D[v, s] = sum_{j,b} onehot(base[v+j])[b] * Q_s[j][b]   (int8 operands, int32 accumulation: no rounding at all)
//      for every start position v of the batch and every (motif, strand) slot s.  Q_s is the exact integer form of the real-valued
//      filter D_real = col0[x0] + sum_{j>=1} w_j[x_j], col0 = w_0 - T'_s rounded up to Float16: Q_s[j][b] = ceil(2^e * entry) + k_j
//      with sum_j k_j = 0, so that D >= 2^e * D_real and "D > 0" is the candidate test (tc_int8_filter in scan.cu).  T'_s = t_s - E_s
//      - eps32 where E_s bounds |Float16 running sum - real sum| over all paths whose Float16 score exceeds t_s (tc_error_bound below:
//      U_j = the Float16 running sum of column maxima bounds every partial sum from above by monotonicity of rounding, a backward
//      recursion bounds the partial sums of hit paths from below, each add errs by at most 2^-11 |partial sum|).  Hence every true
//      hit has D_real > eps32 > 0 and D >= 1; candidates (a few 1e-4 of all cells at the usual thresholds) go to a list in HBM.
//   2. k_scan_tc_verify: one thread per candidate re-computes the sequential Float16 score (same table, same adds as
//      emit_kernel) and sets the bit of the hit mask when score > thresh.  The masks then feed count / emit / hist unchanged, so
//      hit sets are bit-identical to scan_kernel's (tests/test_scan_gpu.py runs both paths on the same inputs).
//
// Operand layout (the im2col matrix is never materialised): a tile is 128 start positions of one phase, v = v0 + ph + 4m, ph < 4.
// Its one-hot stream in shared memory holds one 16-byte chunk per 4 bases (one byte per base and class {A,C,G,T}); row m of the A
// operand is the stream from chunk m on, so in the canonical K-major no-swizzle UMMA layout (core matrix = 8 rows x 16 B, rows 16 B
// apart) the operand of K-chunk c is the same stream advanced by c*16 B.  Two copies ("planes", the second shifted by one chunk)
// give the two K-chunks of one K=32 MMA at LBO = plane stride; SBO = 128 B.  B = Q[K chunk][256 slots][16 bytes] stays resident.
// One CTA per SM owns one or two blocks of 256 slots; warps 0 and 18 build streams (from the 2-bit words in L2), warp 1 (converged, one
// elected lane per instruction) issues kchunks/2 MMAs of 128x256x32 per tile, block and phase, warps 2-17 drain every accumulator use:
// two tcgen05.ld of 32 lanes x 32 columns each, accumulator handed back, then a 3-input max tree; individual columns are looked at only
// when some lane saw a positive value.  "tc_error_bound below" = tc_error_bound() in scan.cu (host).
#pragma once

#define TCS_M 128
#define TCS_N 256                          // slots per block = accumulator columns
#define TCS_PHASES 4                       // start positions v0 + ph + 4m of one tile: 4 phases x 128 rows
#define TCS_TILE (TCS_PHASES * TCS_M)      // start positions per tile
#define TCS_STREAM 160                     // 16-byte chunks per stream plane: 128 rows + up to 16 K-chunks, in the producers' steps of 32
#define TCS_PLANE_BYTES (TCS_STREAM * 16)
#define TCS_STAGE_BYTES (TCS_PHASES * 2 * TCS_PLANE_BYTES)   // one tile: 4 phases x {plane 0, plane 1}
#define TCS_STAGES 4
#define TCS_THREADS 608                    // warps: 0 and 18 producers, 1 MMA issue, 2-17 epilogue
#define TCS_RESERVE 256                    // candidate records reserved per global atomic
#define TCS_MAX_KCHUNKS 16                 // 64 columns x 4 bases / 16
#define TCS_MAX_ENTRIES 16                 // work entries (single or paired slot blocks) per launch: up to 4096 motifs
#ifndef TCS_PROFILE
#define TCS_PROFILE 0                      // 1: per-role wait clocks in TcArgs::dbg (printed with MB200_SCAN_TC_DEBUG=1)
#endif
#if TCS_PROFILE
#define TCS_PROF(...) __VA_ARGS__
#else
#define TCS_PROF(...)
#endif

struct TcBlock {                           // what one CTA works on: one block of 256 slots, or a long and a short block paired
    int64_t b_off[2];                      // byte offsets of the B operands in the TC blob
    int32_t kchunks[2];                    // 16-byte K chunks (16 int8 = 4 PWM columns), even
    int32_t slot0[2];                      // first global slot
    int32_t nsub;                          // 1, or 2: sub-block 0 (the longer one) accumulates in TMEM columns [0,256), sub-block 1 in [256,512)
    int32_t cta0, nctas;                   // CTAs [cta0, cta0 + nctas) work on this entry
    int32_t pad;
};
struct TcSlot {                            // per global slot, for the epilogue (npos) and the verifier
    int32_t motif;                         // original motif index, -1: disabled
    int32_t strand, len, npos;
    uint32_t thr;                          // Float16 bits of max(thresh, 0)
    int32_t pad[3];
};
struct TcArgs {
    const uint32_t* seqw; int64_t rowwords; int64_t seq0;
    const int64_t* lens;                   // ragged stores: row lengths (nullptr: every row has Lb bases)
    uint32_t Lb; uint32_t vtotal;          // virtual positions of the batch: v = n_local * Lb + p
    const uint8_t* blob; int32_t nblocks;
    TcBlock blocks[TCS_MAX_ENTRIES];       // by value: kernel parameters live in the constant bank, so everything derived from an entry (trip
                                           // counts, descriptors) is provably warp-uniform and stays in uniform registers
    const TcSlot* slots;
    unsigned long long* list; unsigned long long cap; unsigned long long* gcount;   // candidate list, its capacity, reserved records
    uint32_t* overflow;
    int32_t ntiles;                        // tiles of TCS_TILE positions (TCS_PHASES units each)
    long long* clocks;                     // [grid][2]: clocks the MMA lane spent on its tiles, tiles done (feeds the host's re-balancing of CTAs over blocks)
    long long* dbg;                        // TCS_PROFILE builds: [grid][8] wait clocks per role
};

__device__ __forceinline__ uint64_t tcs_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // UMMA shared-memory descriptor, K-major, SWIZZLE_NONE: [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// Issued by the whole (converged) MMA warp: one elected lane executes the instruction.  Keeping the warp converged lets the compiler
// hold descriptors, TMEM address and instruction descriptor in uniform registers (no per-MMA R2UR/ELECT sequences).
__device__ __forceinline__ void tcs_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\telect.sync _|q, 0xFFFFFFFF;\n\t@q tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
                 :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tcs_commit(uint32_t bar) {
    asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xFFFFFFFF;\n\t@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void tcs_wait(uint32_t bar, uint32_t parity) {
    uint32_t done, spins = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (!done && ++spins > (1u << 26)) __trap();             // never hang the device on a lost completion
    } while (!done);
}
// one-hot bytes {A,C,G,T} of one base: 4 bases make a 16-byte chunk
__device__ __forceinline__ uint32_t tcs_onehot(uint32_t b) { return 1u << (8 * b); }
__device__ __forceinline__ uint32_t tcs_base(const TcArgs& a, uint32_t v) {
    if (v >= a.vtotal) return 0u;
    const uint32_t n = v / a.Lb, p = v - n * a.Lb;
    const uint32_t w = __ldg(a.seqw + (a.seq0 + n) * a.rowwords + (p >> 4));
    return (w >> ((p & 15) * 2)) & 3u;
}

// A warp's slice of the candidate list is used up: pad it with empty records and reserve the next one (one global atomic per
// TCS_RESERVE records).  ~0: the list is full, the host falls back to scan_kernel for this batch.
__device__ __noinline__ unsigned long long tcs_reserve(unsigned long long* list, unsigned long long* gcount, unsigned long long cap, uint32_t* overflow,
                                                       int lane, unsigned long long cur, unsigned long long end) {
    for (unsigned long long i = cur + lane; i < end; i += 32) list[i] = ~0ull;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(gcount, (unsigned long long)TCS_RESERVE);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base + TCS_RESERVE > cap) {
        if (lane == 0) atomicExch(overflow, 1u);
        return ~0ull;
    }
    return base;
}

#define TCS_LDTM32(U, TADDR)                                                                                                                   \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];" \
                 : "=r"(U[0]), "=r"(U[1]), "=r"(U[2]), "=r"(U[3]), "=r"(U[4]), "=r"(U[5]), "=r"(U[6]), "=r"(U[7]), "=r"(U[8]), "=r"(U[9]), "=r"(U[10]),           \
                   "=r"(U[11]), "=r"(U[12]), "=r"(U[13]), "=r"(U[14]), "=r"(U[15]), "=r"(U[16]), "=r"(U[17]), "=r"(U[18]), "=r"(U[19]), "=r"(U[20]),      \
                   "=r"(U[21]), "=r"(U[22]), "=r"(U[23]), "=r"(U[24]), "=r"(U[25]), "=r"(U[26]), "=r"(U[27]), "=r"(U[28]), "=r"(U[29]), "=r"(U[30]), "=r"(U[31]) \
                 : "r"(TADDR) : "memory")

// max of 32 int32 accumulator values as four independent chains (latency, not issue, bounds the epilogue).  Integer max: read as
// floats, bit patterns >= 0x7F800001 would be NaN and be dropped by max.f32.
__device__ __forceinline__ int tcs_max32(const uint32_t (&u)[32]) {
    int m[4];
    #pragma unroll
    for (int k = 0; k < 4; ++k) {
        m[k] = __vimax3_s32((int)u[8 * k], (int)u[8 * k + 1], (int)u[8 * k + 2]);
        m[k] = __vimax3_s32(m[k], (int)u[8 * k + 3], (int)u[8 * k + 4]);
        m[k] = __vimax3_s32(m[k], (int)u[8 * k + 5], (int)u[8 * k + 6]);
    }
    return max(__vimax3_s32(m[0], m[1], m[2]), __vimax3_s32(m[3], (int)u[7], __vimax3_s32((int)u[15], (int)u[23], (int)u[31])));
}
// bit c set when column c is positive
__device__ __forceinline__ uint32_t tcs_posbits(const uint32_t (&u)[32]) {
    uint32_t b = 0;
    #pragma unroll
    for (int c = 31; c >= 0; --c) b = __funnelshift_l((uint32_t)(-(int32_t)u[c]), b, 1);       // shifts in the sign of -u: set exactly when (int)u > 0
    return b;
}

// Some lane of the warp has a positive column among these 64 (two chunks): append (slot, position) records of every positive
// column.  Windows that run past the end of their sequence are left to the verifier (it knows the motif length).
__device__ __noinline__ void tcs_append(unsigned long long* list, unsigned long long* gcount, unsigned long long cap, uint32_t* overflow, int lane,
                                        uint32_t bits0, uint32_t bits1, uint32_t slot_base, uint32_t v, unsigned long long* cur_end, uint32_t* dead) {
    if (*dead) return;
    const uint32_t cnt = __popc(bits0) + __popc(bits1);
    const uint32_t who = __ballot_sync(0xffffffffu, cnt != 0u);
    uint32_t incl = cnt, total;                                                          // inclusive prefix sum over lanes
    if ((who & (who - 1u)) == 0u) {                                                      // the usual case: one lane has candidates
        total = __shfl_sync(0xffffffffu, cnt, __ffs(who) - 1);
    } else {
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
        total = __shfl_sync(0xffffffffu, incl, 31);
    }
    unsigned long long cur = cur_end[0], end = cur_end[1];
    if (cur + total > end) {
        if (total > TCS_RESERVE) { if (lane == 0) atomicExch(overflow, 1u); *dead = 1u; return; }     // cannot happen: 32 lanes x 64 columns > 256 only at absurd densities
        cur = tcs_reserve(list, gcount, cap, overflow, lane, cur, end);
        if (cur == ~0ull) { *dead = 1u; cur_end[0] = cur_end[1] = 0; return; }
        end = cur + TCS_RESERVE;
    }
    unsigned long long o = cur + (incl - cnt);
    while (bits0) { const int c = __ffs(bits0) - 1; bits0 &= bits0 - 1; list[o++] = ((unsigned long long)(slot_base + c) << 32) | v; }
    while (bits1) { const int c = __ffs(bits1) - 1; bits1 &= bits1 - 1; list[o++] = ((unsigned long long)(slot_base + 32 + c) << 32) | v; }
    cur_end[0] = cur + total; cur_end[1] = end;
}

// The K loop of one accumulator use, fully unrolled per trip count: with compile-time t the descriptors of step t are the first
// ones plus constants (one uniform 64-bit add each); KP = ceil(len / 8) <= 8.  A run-time loop costs ~26 dependent instructions per MMA in the single issuing
// thread (ELECT + seven R2UR per MMA): ~180 clocks per 128-clock MMA, i.e. the issuing thread, not the tensor pipe, set the pace.
template <int KP>
__device__ __forceinline__ void tcs_issue_n(uint32_t tmem_d, uint64_t da0, uint64_t db0, uint32_t idesc) {
    #pragma unroll
    for (int t = 0; t < KP; ++t) tcs_mma(tmem_d, da0 + (uint64_t)(2 * t), db0 + (uint64_t)(2 * t * TCS_N), idesc, t ? 1u : 0u);
}
__device__ __forceinline__ void tcs_issue(int kp, uint32_t tmem_d, uint64_t da0, uint64_t db0, uint32_t idesc) {
    switch (kp) {
        case 1: tcs_issue_n<1>(tmem_d, da0, db0, idesc); break; case 2: tcs_issue_n<2>(tmem_d, da0, db0, idesc); break;
        case 3: tcs_issue_n<3>(tmem_d, da0, db0, idesc); break; case 4: tcs_issue_n<4>(tmem_d, da0, db0, idesc); break;
        case 5: tcs_issue_n<5>(tmem_d, da0, db0, idesc); break; case 6: tcs_issue_n<6>(tmem_d, da0, db0, idesc); break;
        case 7: tcs_issue_n<7>(tmem_d, da0, db0, idesc); break; default: tcs_issue_n<8>(tmem_d, da0, db0, idesc); break;
    }
}

// Work item = one tile of 512 consecutive virtual start positions = four phases (offsets mod 4) of 128 rows.
// Single block: even phases accumulate in TMEM columns [0,256), odd phases in [256,512).
// Paired blocks (nsub = 2): draining 128 x 256 int32 accumulators costs >= 512 clocks of TMEM read bandwidth, more than the MMA
// time of a short block (16 columns: 256 clocks) and far less than that of a long one, so a long and a short block share the CTA
// and the one-hot streams: unit order (long, ph0) (short, ph0) (long, ph1) (short, ph1) ..., long -> accumulator 0, short ->
// accumulator 1; the long block's accumulator drains under the short block's MMAs and vice versa.
// Warps: 0 and 18 build the one-hot streams of alternate tiles, one lane of warp 1 issues the MMAs, warps 2-17 drain the
// accumulators (8 warps each: 4 TMEM lane quarters x 2 column halves).
__global__ void __launch_bounds__(TCS_THREADS, 1) k_scan_tc(const TcArgs a) {
    extern __shared__ __align__(1024) uint8_t tcs_smem[];
    uint8_t* sA = tcs_smem;                                              // [TCS_STAGES][TCS_PHASES][2 planes][TCS_STREAM][16 B]
    uint8_t* sB = tcs_smem + TCS_STAGES * TCS_STAGE_BYTES;               // per sub-block [kchunks][256][16 B]
    __shared__ __align__(8) uint64_t s_bars[2 * TCS_STAGES + 5];         // full[S], empty[S], accfull[2], accempty[2], B landed
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    auto bar = [&](int i) { return (uint32_t)__cvta_generic_to_shared(&s_bars[i]); };

    // which slot block does this CTA serve
    int bi = 0;
    for (int i = 0; i < a.nblocks; ++i) if ((int)blockIdx.x >= a.blocks[i].cta0) bi = i;
    const TcBlock blk = a.blocks[bi];
    const int rank = (int)blockIdx.x - blk.cta0;
    if (rank >= blk.nctas) return;

    if (tid == 0) {
        for (int i = 0; i < 2 * TCS_STAGES + 2; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar(i)) : "memory");
        for (int i = 2 * TCS_STAGES + 2; i < 2 * TCS_STAGES + 4; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 16;" :: "r"(bar(i)) : "memory");   // all 16 epilogue warps drain every accumulator use
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar(2 * TCS_STAGES + 4)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"((uint32_t)__cvta_generic_to_shared(&s_tmem)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // the last chunk of every shifted plane is never written by the producers (and never needed): keep it zero
    for (int i = tid; i < TCS_STAGES * TCS_PHASES; i += blockDim.x)
        *reinterpret_cast<uint4*>(sA + (size_t)i * (2 * TCS_PLANE_BYTES) + TCS_PLANE_BYTES + (TCS_STREAM - 1) * 16) = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = s_tmem;
    const uint32_t sA_addr = (uint32_t)__cvta_generic_to_shared(sA), sB_addr = (uint32_t)__cvta_generic_to_shared(sB);
    // instruction descriptor: D = S32 (2<<4), A and B signed 8-bit (1<<7, 1<<10), both K-major, N>>3 at bit 17, M>>4 at bit 24
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TCS_N >> 3) << 17) | ((uint32_t)(TCS_M >> 4) << 24);

    if (warp == 0 || warp == TCS_THREADS / 32 - 1) {
        // ---- producers: bases v0 .. v0+642 of the tile -> the stream of phase f, S_f[m] = (b[4m+f], .., b[4m+f+3]), stored twice
        //      (plane 1 = plane 0 shifted by one chunk) ----
        const int pw = warp == 0 ? 0 : 1;
        TCS_PROF(long long w_prod = 0;)
        int it = 0;
        for (int tile = rank; tile < a.ntiles; tile += blk.nctas, ++it) {
            if ((it & 1) != pw) continue;
            const int st = it % TCS_STAGES; const uint32_t ph = (it / TCS_STAGES) & 1;
            uint32_t v = (uint32_t)tile * TCS_TILE + 4u * lane;
            uint32_t n = v / a.Lb, p = v - n * a.Lb;
            const uint32_t* row = a.seqw + (a.seq0 + n) * a.rowwords;
            uint32_t bb[TCS_STREAM / 32];                                                // bases 4m .. 4m+3 of chunk m = lane + 32 i, 2 bits each
            #pragma unroll
            for (int i = 0; i < TCS_STREAM / 32; ++i) {
                bb[i] = 0;
                #pragma unroll
                for (int k = 0; k < 4; ++k) {
                    uint32_t pk = p + k; const uint32_t* rk = row;
                    while (pk >= a.Lb) { pk -= a.Lb; rk += a.rowwords; }
                    const uint32_t w = v + k < a.vtotal ? __ldg(rk + (pk >> 4)) : 0u;
                    bb[i] |= ((w >> ((pk & 15) * 2)) & 3u) << (2 * k);
                }
                v += 128; p += 128;
                while (p >= a.Lb) { p -= a.Lb; row += a.rowwords; }
            }
            TCS_PROF(const long long t0 = clock64();)
            tcs_wait(bar(TCS_STAGES + st), ph ^ 1);                                      // stage free
            TCS_PROF(w_prod += clock64() - t0;)
            uint8_t* s0 = sA + (size_t)st * TCS_STAGE_BYTES;                             // phase f: plane 0 at s0 + 2f planes, plane 1 after it
            #pragma unroll
            for (int i = 0; i < TCS_STREAM / 32; ++i) {
                const uint32_t m = lane + 32 * i;
                uint32_t nb = __shfl_down_sync(0xffffffffu, bb[i], 1);                    // bases 4m+4 .. 4m+7: the next chunk's
                const uint32_t nxt = __shfl_sync(0xffffffffu, i + 1 < TCS_STREAM / 32 ? bb[(i + 1) % (TCS_STREAM / 32)] : 0u, 0);
                if (lane == 31) nb = nxt;
                const uint32_t b7 = bb[i] | (nb << 8);
                uint32_t o[7];                                                           // one-hot of bases 4m .. 4m+6
                #pragma unroll
                for (int k = 0; k < 7; ++k) o[k] = tcs_onehot((b7 >> (2 * k)) & 3u);
                #pragma unroll
                for (int f = 0; f < TCS_PHASES; ++f) {
                    const uint4 c = make_uint4(o[f], o[f + 1], o[f + 2], o[f + 3]);
                    uint8_t* pl = s0 + (size_t)f * 2 * TCS_PLANE_BYTES;
                    *reinterpret_cast<uint4*>(pl + m * 16) = c;
                    if (m > 0) *reinterpret_cast<uint4*>(pl + TCS_PLANE_BYTES + (m - 1) * 16) = c;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");                 // generic-proxy writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar(st)) : "memory");
        }
        TCS_PROF(if (a.dbg && warp == 0 && lane == 0) a.dbg[blockIdx.x * 8 + 5] = w_prod;)
    } else if (warp == 1) {
        {   // ---- MMA warp: all 32 lanes run this code converged; tcs_mma / tcs_commit elect the issuing lane ----
            const uint32_t b_bytes0 = (uint32_t)blk.kchunks[0] * TCS_N * 16;
            if (lane == 0) {   // the B operands, resident for the whole kernel
                const uint32_t b_bytes1 = blk.nsub > 1 ? (uint32_t)blk.kchunks[1] * TCS_N * 16 : 0u;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar(2 * TCS_STAGES + 4)), "r"(b_bytes0 + b_bytes1) : "memory");
                for (int sub = 0; sub < blk.nsub; ++sub) {
                    const uint32_t nbytes = sub ? b_bytes1 : b_bytes0, dst = sB_addr + (sub ? b_bytes0 : 0u);
                    for (uint32_t o = 0; o < nbytes; o += 32768u) {
                        const uint32_t nb = min(32768u, nbytes - o);
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     :: "r"(dst + o), "l"(a.blob + blk.b_off[sub] + o), "r"(nb), "r"(bar(2 * TCS_STAGES + 4)) : "memory");
                    }
                }
            }
            tcs_wait(bar(2 * TCS_STAGES + 4), 0);
            const uint64_t dbA = tcs_desc(sB_addr, TCS_N * 16, 128), dbB = tcs_desc(sB_addr + b_bytes0, TCS_N * 16, 128);
            const int kpA = blk.kchunks[0] >> 1, kpB = blk.kchunks[1] >> 1;
            TCS_PROF(long long w_full = 0; long long w_acc = 0;)
            const long long t_start = clock64();
            uint32_t use0 = 0, use1 = 0;                                                 // completed uses of each accumulator
            int it = 0;
            for (int tile = rank; tile < a.ntiles; tile += blk.nctas, ++it) {
                const int st = it % TCS_STAGES; const uint32_t ph = (it / TCS_STAGES) & 1;
                TCS_PROF(long long t0 = clock64();)
                tcs_wait(bar(st), ph);                                                   // streams built
                TCS_PROF(w_full += clock64() - t0;)
                #pragma unroll
                for (int f = 0; f < TCS_PHASES; ++f) {
                    for (int sub = 0; sub < blk.nsub; ++sub) {
                        const int ac = blk.nsub > 1 ? sub : (f & 1);
                        const uint32_t uses = ac ? use1 : use0;
                        TCS_PROF(t0 = clock64();)
                        tcs_wait(bar(2 * TCS_STAGES + 2 + ac), (uses & 1) ^ 1);          // accumulator drained
                        TCS_PROF(w_acc += clock64() - t0;)
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint64_t da0 = tcs_desc(sA_addr + st * TCS_STAGE_BYTES + f * 2 * TCS_PLANE_BYTES, TCS_PLANE_BYTES, 128);
                        const uint64_t dbs = sub ? dbB : dbA;
                        const int kp = sub ? kpB : kpA;
                        tcs_issue(kp, tmem + ac * TCS_N, da0, dbs, idesc);
                        tcs_commit(bar(2 * TCS_STAGES + ac));
                        if (ac) ++use1; else ++use0;
                    }
                }
                tcs_commit(bar(TCS_STAGES + st));
            }
            if (a.clocks && lane == 0) { a.clocks[blockIdx.x * 2] = clock64() - t_start; a.clocks[blockIdx.x * 2 + 1] = it; }
            TCS_PROF(if (a.dbg && lane == 0) { a.dbg[blockIdx.x * 8 + 0] = clock64() - t_start; a.dbg[blockIdx.x * 8 + 1] = w_full; a.dbg[blockIdx.x * 8 + 2] = w_acc; a.dbg[blockIdx.x * 8 + 6] = bi; a.dbg[blockIdx.x * 8 + 7] = it; })
        }
    } else {
        // ---- epilogue: 16 warps = {TMEM lane quarter} x {64-column group}; every warp drains its 32 lanes x 64 columns of EVERY
        //      accumulator use, in the MMA warp's order.  Both tcgen05.ld of a use are issued before the first wait: with four warps
        //      per SM sub-partition that keeps ~32 KB of TMEM reads in flight (the loads, ~200 clocks of latency each, not the
        //      reduction, bound the drain) ----
        const int q = warp & 3;                                                          // TMEM lane quarter = warp id % 4
        const int cg = (warp - 2) >> 2;                                                  // column group
        unsigned long long cur_end[2] = {0, 0};                                          // this warp's reserved slice of the candidate list
        uint32_t dead = 0;                                                               // list capacity exhausted
        TCS_PROF(long long w_epi = 0; const long long t_start = clock64();)
        uint32_t use0 = 0, use1 = 0;                                                     // completed uses of each accumulator
        int it = 0;
        for (int tile = rank; tile < a.ntiles; tile += blk.nctas, ++it)
        #pragma unroll 1
        for (int f = 0; f < TCS_PHASES; ++f)
        for (int sub = 0; sub < blk.nsub; ++sub) {
            const int ac = blk.nsub > 1 ? sub : (f & 1);
            const uint32_t uses = ac ? use1 : use0;
            if (ac) ++use1; else ++use0;
            const uint32_t v = (uint32_t)tile * TCS_TILE + (uint32_t)f + 4u * (uint32_t)(q * 32 + lane);
            const bool inb = v < a.vtotal;
            TCS_PROF(const long long t0 = clock64();)
            tcs_wait(bar(2 * TCS_STAGES + ac), uses & 1);
            TCS_PROF(w_epi += clock64() - t0;)
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t taddr = tmem + ac * TCS_N + cg * 64 + ((uint32_t)(q * 32) << 16);
            uint32_t ua[32], ub[32];
#ifdef TCS_EXPERIMENT_NO_DRAIN        // timing experiment only: the accumulator is handed back without being read (pure hand-off latency)
            #pragma unroll
            for (int i = 0; i < 32; ++i) ua[i] = 0x80000000u + taddr;
#else
            TCS_LDTM32(ua, taddr);
#endif
#if defined(TCS_EXPERIMENT_HALF_DRAIN) || defined(TCS_EXPERIMENT_NO_DRAIN)      // timing experiment only (results are wrong): read half of the accumulator columns
            #pragma unroll
            for (int i = 0; i < 32; ++i) ub[i] = ua[i];
#else
            TCS_LDTM32(ub, taddr + 32);
#endif
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar(2 * TCS_STAGES + 2 + ac)) : "memory");    // the values are in registers: the accumulator may be overwritten
            const int ma = tcs_max32(ua), mb = tcs_max32(ub);
            bool pos = inb && max(ma, mb) > 0;
            if (__any_sync(0xffffffffu, pos)) {          /* about one use in ten at the usual thresholds */
                // ragged store: a start position in the row's zero padding (poly-A) is no candidate, or an A-rich PWM would fill the
                // list with padding.  Windows that start inside the row and run into the padding are left to the verifier.
                bool live = inb;
                if (a.lens) {
                    const uint32_t n = v / a.Lb;
                    live = inb && (int64_t)(v - n * a.Lb) < __ldg(a.lens + a.seq0 + n);
                    pos = pos && live;
                }
                if (!a.lens || __any_sync(0xffffffffu, pos)) {
                    uint32_t cb0 = 0u, cb1 = 0u;             // bit masks of the positive columns, only for the chunk(s) that have any
                    if (__any_sync(0xffffffffu, live && ma > 0)) cb0 = pos ? tcs_posbits(ua) : 0u;
                    if (__any_sync(0xffffffffu, live && mb > 0)) cb1 = pos ? tcs_posbits(ub) : 0u;
                    tcs_append(a.list, a.gcount, a.cap, a.overflow, lane, cb0, cb1, (uint32_t)(blk.slot0[sub] + cg * 64), v, cur_end, &dead);
                }
            }
        }
        for (unsigned long long i = cur_end[0] + lane; i < cur_end[1]; i += 32) a.list[i] = ~0ull;
        TCS_PROF(if (a.dbg && warp == 2 && lane == 0) { a.dbg[blockIdx.x * 8 + 3] = w_epi; a.dbg[blockIdx.x * 8 + 4] = clock64() - t_start; })
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "n"(512) : "memory");
}

// Exact re-scoring of the candidates: the sequential Float16 adds of greedy_search!, then score > thresh sets the mask bit.
__global__ void __launch_bounds__(256) k_scan_tc_verify(const unsigned long long* __restrict__ list, const unsigned long long* __restrict__ gcount,
                                                        unsigned long long cap, const TcSlot* __restrict__ slots, const EmitMotif* __restrict__ em,
                                                        const uint8_t* __restrict__ blob, const uint32_t* __restrict__ seqw, int64_t rowwords, int64_t seq0,
                                                        uint32_t Lb, int32_t W, int32_t K2pad, uint32_t* __restrict__ mask, unsigned long long* __restrict__ stats,
                                                        uint32_t* __restrict__ unit_bits, uint32_t* __restrict__ unit_list, unsigned long long* __restrict__ n_units,
                                                        const int64_t* __restrict__ lens) {
    if (gcount[1]) return;                                                                // the list overflowed: this batch is re-run on scan_kernel
    const unsigned long long total = min(*gcount, cap);
    unsigned int n_cand = 0, n_hit = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long rec = list[i];
        if (rec == ~0ull) continue;
        const uint32_t slot = (uint32_t)(rec >> 32), v = (uint32_t)rec;
        const uint32_t n = v / Lb, p = v - n * Lb;
        const TcSlot sl = slots[slot];
        if ((int32_t)p >= sl.npos) continue;                                              // the window runs past the end of its sequence (or the slot is disabled)
        if (lens && (int64_t)p + sl.len > lens[seq0 + n]) continue;                       // ragged store: ... past the end of its own row
        const EmitMotif m = em[sl.motif];
        const uint8_t* tab = blob + m.tab_off + sl.strand * m.strand_stride;
        const uint32_t* srow = seqw + (seq0 + n) * rowwords;
        __half s = __ushort_as_half((unsigned short)0);
        for (int32_t j = 0; j < sl.len; ++j) {
            const uint32_t qq = p + j;
            const uint32_t base = (__ldg(srow + (qq >> 4)) >> ((qq & 15) * 2)) & 3u;
            s = __hadd(s, *reinterpret_cast<const __half*>(tab + (int64_t)j * m.col_stride + base * m.base_stride));
        }
        ++n_cand;
        if (__hgt(s, __ushort_as_half((unsigned short)sl.thr))) {
            atomicOr(&mask[((int64_t)n * W + (p >> 5)) * (int64_t)K2pad + slot], 1u << (p & 31));
            ++n_hit;
            if (unit_bits) {                                                              // first hit of this (sequence, motif) unit: list it for count_listed_kernel
                const uint32_t g = n * (uint32_t)(K2pad >> 1) + (slot >> 1);
                const uint32_t bit = 1u << (g & 31);
                if (!(atomicOr(&unit_bits[g >> 5], bit) & bit)) unit_list[atomicAdd(n_units, 1ull)] = g;
            }
        }
    }
    if (stats) {
        n_cand = __reduce_add_sync(0xffffffffu, n_cand);
        n_hit = __reduce_add_sync(0xffffffffu, n_hit);
        if ((threadIdx.x & 31) == 0 && n_cand) { atomicAdd(&stats[0], (unsigned long long)n_cand); atomicAdd(&stats[1], (unsigned long long)n_hit); }
    }
}
