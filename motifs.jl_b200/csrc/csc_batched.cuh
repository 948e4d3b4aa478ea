// Batched-shape variants of the three D/F-layer forms that dominate code retrieval and many-group steps.
//
// The kernels in csc_kernels.cuh are laid out for ONE reference batch (6 sequences): one warp or one block per output
// element, so that a 6-sequence step exposes enough parallelism to hide latency.  With hundreds of groups per launch that
// layout re-reads every operand row from L1/L2 once per output that touches it (k_recon: each (n,p) row of Z,Y 32 times;
// ncu, 500 groups: k_recon 1.36 ms, k_tconv_l 1.03 ms, k_corr_sig 0.55 ms of a 3.4 ms pass).  Here one CTA owns one sequence,
// stages its operands in shared memory once and works on register tiles:
//   k_recon_b     T1  U[p][k] = sum_m a[p][m] F[k][m] + b[p][m] F[f_len-1-k][m]  (a [c x 2M].[2M x 32] product, 4x4 register
//                     tiles), then the overlap-add  out[t] = sum_{p} U[p][t-4p]                       (model.jl:238-239,276-277,313-314)
//   k_corr_sig_b  T2  oa[p][m] = sum_k r[4p+k] F[k][m], ob[p][m] = sum_k r[4p+k] F[f_len-1-k][m]      (model.jl:240-241)
//   k_tconv_b     U1  fx[i+a][j] += x[i][k] F[a][j][k] over the sequence's non-zero codes, scattered into a shared-memory tile
//                     in list order (the same order of additions per output as k_tconv_l)              (model.jl:229,263,294,316,370)
// Same operands, same results up to fp32 summation order (tests compare both layouts).
#pragma once
#include "csc_kernels.cuh"

#define RB_THREADS 256
#define RB_ROUNDS 4              // register tiles a k_recon_b thread may hold: c <= 512 code positions

__device__ __forceinline__ void cp_async8(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
// dynamic shared memory: a,b [cpad][M] (after the products: U [cpad][33]) | FT, FrT [M][32].  The code rows arrive by asynchronous 8-byte copies
// (a load + store loop paid an L2 round trip per two elements: most of the kernel's time), U re-uses their space, so two CTAs fit an SM and
// one's fill overlaps the other's products.
__global__ void __launch_bounds__(RB_THREADS) k_recon_b(const float* __restrict__ ca, const float* __restrict__ cb,
                                                        const float* __restrict__ filt, int64_t filt_gs,
                                                        float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float rb_smem[];
    const int cpad = (d.c + 3) & ~3;
    float* sa = rb_smem;                          // [cpad][M]
    float* sb = sa + cpad * d.M;
    float* sFT = sb + cpad * d.M;                 // [M][32]: sFT[m][k] = F[k][m]
    float* sFr = sFT + d.M * 32;                  // [M][32]: sFr[m][k] = F[f_len-1-k][m]
    float* sU = rb_smem;                          // [cpad][33], over a/b once every product is in registers
    const int64_t n = blockIdx.x;
    const float* F = filt + (n / d.B) * filt_gs;
    const float* za = ca + n * d.c * d.M;
    const float* zb = cb + n * d.c * d.M;
    const int E = d.c * d.M;
    if ((((uintptr_t)za | (uintptr_t)zb) & 7) == 0 && (E & 1) == 0) {
        for (int e = 2 * threadIdx.x; e < E; e += 2 * RB_THREADS) { cp_async8(sa + e, za + e); cp_async8(sb + e, zb + e); }
        asm volatile("cp.async.commit_group;" ::: "memory");
        for (int e = E + threadIdx.x; e < cpad * d.M; e += RB_THREADS) { sa[e] = 0.f; sb[e] = 0.f; }
    } else {
        for (int e = threadIdx.x; e < cpad * d.M; e += RB_THREADS) { sa[e] = e < E ? za[e] : 0.f; sb[e] = e < E ? zb[e] : 0.f; }
    }
    for (int e = threadIdx.x; e < d.f_len * d.M; e += RB_THREADS) {
        const int k = e / d.M, m = e - k * d.M;
        const float f = F[e];
        sFT[m * 32 + k] = f; sFr[m * 32 + (d.f_len - 1 - k)] = f;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    // register tiles: 4 positions x 4 taps; a warp holds 4 position tiles x 8 tap tiles, so every operand load is one wavefront.
    // A thread holds up to RB_ROUNDS tiles (c <= 128 * RB_ROUNDS) until all products are done and U may overwrite a, b.
    const int ntile = (cpad >> 2) * 8;
    float u[RB_ROUNDS][4][4];
    #pragma unroll
    for (int rd = 0; rd < RB_ROUNDS; ++rd) {
        const int tile = threadIdx.x + rd * RB_THREADS;
        #pragma unroll
        for (int i = 0; i < 4; ++i)
            #pragma unroll
            for (int j = 0; j < 4; ++j) u[rd][i][j] = 0.f;
        if (tile < ntile) {
            const int pt = tile >> 3, kt = tile & 7;
            const float* a0 = sa + (pt * 4) * d.M;
            const float* b0 = sb + (pt * 4) * d.M;
            #pragma unroll 2
            for (int m = 0; m < d.M; ++m) {
                const float4 f = *reinterpret_cast<const float4*>(sFT + m * 32 + kt * 4);
                const float4 g = *reinterpret_cast<const float4*>(sFr + m * 32 + kt * 4);
                #pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float av = a0[i * d.M + m], bv = b0[i * d.M + m];
                    u[rd][i][0] += av * f.x + bv * g.x; u[rd][i][1] += av * f.y + bv * g.y;
                    u[rd][i][2] += av * f.z + bv * g.z; u[rd][i][3] += av * f.w + bv * g.w;
                }
            }
        }
    }
    __syncthreads();
    #pragma unroll
    for (int rd = 0; rd < RB_ROUNDS; ++rd) {
        const int tile = threadIdx.x + rd * RB_THREADS;
        if (tile < ntile) {
            const int pt = tile >> 3, kt = tile & 7;
            #pragma unroll
            for (int i = 0; i < 4; ++i)
                #pragma unroll
                for (int j = 0; j < 4; ++j) sU[(pt * 4 + i) * 33 + kt * 4 + j] = u[rd][i][j];
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < d.L4; t += RB_THREADS) {
        const int p_hi = min(d.c - 1, t >> 2);
        const int p_lo = max(0, (t - d.f_len + 4) >> 2);
        float acc = 0.f;
        for (int p = p_lo; p <= p_hi; ++p) acc += sU[p * 33 + (t - 4 * p)];
        float* o = out + n * d.L4 + t;
        if (accumulate) *o += acc; else *o = acc;
    }
}
static inline size_t recon_b_smem(const CscDims& d) {
    const size_t cpad = (size_t)((d.c + 3) & ~3);
    return (std::max(2 * cpad * d.M, cpad * 33) + 2 * (size_t)d.M * 32) * 4;
}
static inline bool recon_b_fits(const CscDims& d) { return ((d.c + 3) >> 2) * 8 <= RB_ROUNDS * RB_THREADS; }

// dynamic shared memory: r [L4 + f_len] | F [f_len][Mp], Mp = M rounded up to a multiple of 4
__global__ void __launch_bounds__(RB_THREADS) k_corr_sig_b(const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                                           const float* __restrict__ filt, int64_t filt_gs,
                                                           float* __restrict__ oa, float* __restrict__ ob, int accumulate, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float rb_smem[];
    const int Mp = (d.M + 3) & ~3;
    const int rlen = (d.L4 + d.f_len + 3) & ~3;
    float* sr = rb_smem;                          // [rlen] signal with the one-hot folded in, zero tail
    float* sF = sr + rlen;                        // [f_len][Mp]
    const int64_t n = blockIdx.x;
    const float* F = filt + (n / d.B) * filt_gs;
    for (int t = threadIdx.x; t < rlen; t += RB_THREADS) sr[t] = t < d.L4 ? sig_at(sig, bases, sgn, n, t, d) : 0.f;
    for (int e = threadIdx.x; e < d.f_len * Mp; e += RB_THREADS) {
        const int k = e / Mp, m = e - k * Mp;
        sF[e] = m < d.M ? F[k * d.M + m] : 0.f;
    }
    __syncthreads();
    const int cpad = (d.c + 3) & ~3, mt_n = Mp >> 2;
    const int ntile = (cpad >> 2) * mt_n;
    for (int tile = threadIdx.x; tile < ntile; tile += RB_THREADS) {
        const int pt = tile / mt_n, mt = tile - pt * mt_n;
        float a[4][4], b[4][4];
        #pragma unroll
        for (int i = 0; i < 4; ++i)
            #pragma unroll
            for (int j = 0; j < 4; ++j) { a[i][j] = 0.f; b[i][j] = 0.f; }
        const float* r0 = sr + 16 * pt;            // position p = 4pt+i reads r[4p + k] = r0[4i + k]
        #pragma unroll 4
        for (int k = 0; k < d.f_len; ++k) {
            const float4 f = *reinterpret_cast<const float4*>(sF + k * Mp + mt * 4);
            const float4 g = *reinterpret_cast<const float4*>(sF + (d.f_len - 1 - k) * Mp + mt * 4);
            #pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float rv = r0[4 * i + k];
                a[i][0] += rv * f.x; a[i][1] += rv * f.y; a[i][2] += rv * f.z; a[i][3] += rv * f.w;
                b[i][0] += rv * g.x; b[i][1] += rv * g.y; b[i][2] += rv * g.z; b[i][3] += rv * g.w;
            }
        }
        const bool pairs = (d.M & 1) == 0 && (((uintptr_t)oa | (uintptr_t)ob) & 7) == 0;      // 8-byte stores: row starts and tile starts are even
        #pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int p = pt * 4 + i;
            if (p >= d.c) continue;
            if (pairs) {
                #pragma unroll
                for (int j = 0; j < 4; j += 2) {
                    const int m = mt * 4 + j;
                    if (m >= d.M) continue;
                    float2* pa = reinterpret_cast<float2*>(oa + (n * d.c + p) * d.M + m);
                    float2* pb = reinterpret_cast<float2*>(ob + (n * d.c + p) * d.M + m);
                    float2 va = make_float2(a[i][j], a[i][j + 1]), vb = make_float2(b[i][j], b[i][j + 1]);
                    if (accumulate) { const float2 qa = *pa, qb = *pb; va.x += qa.x; va.y += qa.y; vb.x += qb.x; vb.y += qb.y; }
                    *pa = va; *pb = vb;
                }
                continue;
            }
            #pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int m = mt * 4 + j;
                if (m >= d.M) continue;
                const int64_t o = (n * d.c + p) * d.M + m;
                if (accumulate) { oa[o] += a[i][j]; ob[o] += b[i][j]; } else { oa[o] = a[i][j]; ob[o] = b[i][j]; }
            }
        }
    }
}
static inline size_t corr_sig_b_smem(const CscDims& d) {
    const size_t Mp = (size_t)((d.M + 3) & ~3), rlen = (size_t)((d.L4 + d.f_len + 3) & ~3);
    return (rlen + (size_t)d.f_len * Mp) * 4;
}

// F [h][2M][K] -> Ft [K][h*2M] (per group when gs != 0): the tap rows of one syntax filter become contiguous
__global__ void __launch_bounds__(256) k_transpose_F(const float* __restrict__ F, int64_t gs, float* __restrict__ Ft, int G, CscDims d) { PDL_SYNC();
    const int hj = d.h * d.M2;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)G * hj * d.K) return;
    const int k = (int)(t % d.K);
    const int64_t r = t / d.K;
    const int e = (int)(r % hj);
    const int64_t g = r / hj;
    Ft[(g * d.K + k) * hj + e] = F[g * gs + (int64_t)e * d.K + k];
}

#define TB_PF 4                     // codes whose filter rows a k_tconv_b thread holds ahead
#define TB_E 5                      // window offsets per thread: h * 2M <= 1280
// dynamic shared memory: tile [c][2M].  Ft as written by k_transpose_F (ft_gs = K*h*2M per group, or 0 when shared).
__global__ void __launch_bounds__(RB_THREADS) k_tconv_b(const float* __restrict__ x, const int32_t* __restrict__ lcnt, const uint16_t* __restrict__ lidx,
                                                        const float* __restrict__ lval, const float* __restrict__ Ft, int64_t ft_gs,
                                                        float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float rb_smem[];
    float* tile = rb_smem;
    __shared__ int s_i[LIST_CAP], s_k[LIST_CAP];
    __shared__ float s_v[LIST_CAP];
    const int64_t n = blockIdx.x;
    const float* FT = Ft + (n / d.B) * ft_gs;
    const int hj = d.h * d.M2, E = d.c * d.M2;
    const int cnt = lcnt[n];
    for (int e = threadIdx.x; e < E; e += RB_THREADS) tile[e] = 0.f;
    if (cnt <= LIST_CAP && threadIdx.x < cnt) {
        const int e = lidx[n * LIST_CAP + threadIdx.x];
        s_i[threadIdx.x] = e / d.K; s_k[threadIdx.x] = e % d.K; s_v[threadIdx.x] = lval[n * LIST_CAP + threadIdx.x];
    }
    __syncthreads();
    if (cnt <= LIST_CAP && hj <= TB_E * RB_THREADS) {
        // rows i..i+h-1 of the tile are one contiguous window of h*2M floats: window[e] += v * Ft[k][e].  The filter rows of the next TB_PF codes
        // are already in registers when a code's turn comes: with the load behind the block barrier of the previous code the kernel was a chain
        // of ~32 L2 round trips per sequence.
        float fb[TB_PF][TB_E];
        #pragma unroll
        for (int u = 0; u < TB_PF; ++u)
            #pragma unroll
            for (int r = 0; r < TB_E; ++r) { const int e = threadIdx.x + r * RB_THREADS; fb[u][r] = (u < cnt && e < hj) ? FT[(int64_t)s_k[u] * hj + e] : 0.f; }
        for (int q0 = 0; q0 < cnt; q0 += TB_PF) {
            #pragma unroll
            for (int u = 0; u < TB_PF; ++u) {
                const int q = q0 + u;
                if (q < cnt) {                     // block-uniform
                    float* w = tile + s_i[q] * d.M2;
                    const float v = s_v[q];
                    #pragma unroll
                    for (int r = 0; r < TB_E; ++r) { const int e = threadIdx.x + r * RB_THREADS; if (e < hj) w[e] += v * fb[u][r]; }
                    if (q + TB_PF < cnt) {
                        #pragma unroll
                        for (int r = 0; r < TB_E; ++r) { const int e = threadIdx.x + r * RB_THREADS; if (e < hj) fb[u][r] = FT[(int64_t)s_k[q + TB_PF] * hj + e]; }
                    }
                    __syncthreads();               // the next code's window overlaps this one with other threads
                }
            }
        }
    } else if (cnt <= LIST_CAP) {
        for (int q = 0; q < cnt; ++q) {
            float* w = tile + s_i[q] * d.M2;
            const float* f = FT + (int64_t)s_k[q] * hj;
            const float v = s_v[q];
            for (int e = threadIdx.x; e < hj; e += RB_THREADS) w[e] += v * f[e];
            __syncthreads();
        }
    } else {                                       // more than LIST_CAP non-zeros: walk x itself in the same (position, filter) order
        const float* xr = x + n * d.l * d.K;
        for (int q = 0; q < d.l * d.K; ++q) {
            const float v = xr[q];
            if (v == 0.f) continue;                // block-uniform
            float* w = tile + (q / d.K) * d.M2;
            const float* f = FT + (int64_t)(q % d.K) * hj;
            for (int e = threadIdx.x; e < hj; e += RB_THREADS) w[e] += v * f[e];
            __syncthreads();
        }
    }
    float* o = out + n * E;
    for (int e = threadIdx.x; e < E; e += RB_THREADS) { if (accumulate) o[e] += tile[e]; else o[e] = tile[e]; }
}

// A4 for many groups: one CTA per group, the same order-statistic scheme as k_mask_scale_c (one 4096-bin level on bits 30..19,
// then the few hundred entries of the median's bin resolved in shared memory) but with the group's 2*B*c*M values re-read from
// L2 in each of the three sweeps instead of being held in shared memory: 24 KB of shared memory per CTA, two CTAs per SM, and
// no cap on the group size.  (k_mask_scale_s keeps up to 49 152 positives in shared memory and runs four 8-bit radix passes over
// them with one CTA per SM: 304 us per 500 groups; this kernel: see profiles/.)
#define MG_THREADS 1024
#ifndef MG_MINB
#define MG_MINB 1                   // CTAs per SM the register allocation of k_mask_scale_g is held to.  2 (32 registers, ~100 bytes of spills) measured: 135 vs 145 us per call at 500 groups x 100 bp, but 9.19 vs 9.11 ms per 64-group step at 200 bp (64 CTAs: occupancy is not the limit there)
#endif
__global__ void __launch_bounds__(MG_THREADS, MG_MINB) k_mask_scale_g(const float* __restrict__ z, const float* __restrict__ y,
                                                             float* __restrict__ zy, float* __restrict__ med_out, CscDims d) { PDL_SYNC();
    __shared__ unsigned int hist[MS_BINS];
    __shared__ float cand[MS_CAND];
    __shared__ unsigned int s_ncand, s_min, wsum[32], res[4];
    const int g = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const int EZ = d.B * d.c * d.M;
    const float* zg = z + (int64_t)g * EZ;
    const float* yg = y + (int64_t)g * EZ;
    const int E2 = 2 * EZ;
    // 16-byte sweeps when a group's slab is a whole number of float4 (27 900 floats at Lb = 100): the sweeps are bound by loads in flight
    const int VZ = (EZ & 3) ? 0 : EZ >> 2, V2 = 2 * VZ;
    const float4* zg4 = reinterpret_cast<const float4*>(zg);
    const float4* yg4 = reinterpret_cast<const float4*>(yg);
    unsigned int prefix = 0, pmask = 0, krank = 0, npos = 0, cnt = 0;
    int shift = 19, nb = MS_BINS;
    bool first = true, resolved = false;
    for (int lvl = 0; lvl < 3; ++lvl) {
        for (int i = threadIdx.x; i < nb; i += MG_THREADS) hist[i] = 0;
        if (threadIdx.x == 0) { s_ncand = 0; s_min = 0x7f800000u; }
        __syncthreads();
        #pragma unroll 4
        for (int v = threadIdx.x; v < V2; v += MG_THREADS) {
            const float4 f4 = v < VZ ? zg4[v] : yg4[v - VZ];
            const float fv[4] = {f4.x, f4.y, f4.z, f4.w};
            #pragma unroll
            for (int i = 0; i < 4; ++i) {
                const unsigned int b = __float_as_uint(fv[i]);
                if (fv[i] > 0.f && (b & pmask) == prefix) atomicAdd(&hist[(b >> shift) & (unsigned)(nb - 1)], 1u);
            }
        }
        for (int e = 4 * V2 + threadIdx.x; e < E2; e += MG_THREADS) {          // group sizes that are not a multiple of 4: scalar sweep
            const float f = e < EZ ? zg[e] : yg[e - EZ];
            const unsigned int b = __float_as_uint(f);
            if (f > 0.f && (b & pmask) == prefix) atomicAdd(&hist[(b >> shift) & (unsigned)(nb - 1)], 1u);
        }
        __syncthreads();
        block_find_bin(hist, nb, krank, first, wsum, res);
        if (first) {
            npos = res[3];
            if (npos == 0) break;
            krank = (npos & 1u) ? npos / 2 : npos / 2 - 1;
            first = false;
        }
        const unsigned int bin = res[0];
        krank -= res[1]; cnt = res[2];
        prefix |= bin << shift; pmask |= (unsigned)(nb - 1) << shift;
        __syncthreads();
        if (cnt <= MS_CAND) break;
        if (shift == 0) { resolved = true; break; }
        if (shift == 19) { shift = 7; nb = MS_BINS; } else { shift = 0; nb = 128; }
    }
    float med = -INFINITY;
    if (npos > 0) {
        // the bin's entries -> cand[], and the smallest entry above the bin
        unsigned int mn = 0x7f800000u;
        auto take = [&](float f) {                                  // candidates are rare (a few hundred of 55 800): plain atomics
            const unsigned int b = __float_as_uint(f);
            if (f > 0.f) {
                if ((b & pmask) > prefix) mn = min(mn, b);
                else if (!resolved && (b & pmask) == prefix) cand[atomicAdd(&s_ncand, 1u)] = f;
            }
        };
        #pragma unroll 4
        for (int v = threadIdx.x; v < V2; v += MG_THREADS) {
            const float4 f4 = v < VZ ? zg4[v] : yg4[v - VZ];
            take(f4.x); take(f4.y); take(f4.z); take(f4.w);
        }
        for (int e = 4 * V2 + threadIdx.x; e < E2; e += MG_THREADS) take(e < EZ ? zg[e] : yg[e - EZ]);
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(FULLMASK, mn, o));
        if (lane == 0 && mn != 0x7f800000u) atomicMin(&s_min, mn);
        __syncthreads();
        const unsigned int kin = krank;
        unsigned int v1b = prefix;
        if (!resolved) {
            unsigned int lowfix = 0, lowmask = 0;
            int rem = shift;
            while (rem > 0) {
                const int nbits = rem < 10 ? rem : 10, sh = rem - nbits, nbin = 1 << nbits;
                for (int i = threadIdx.x; i < nbin; i += MG_THREADS) hist[i] = 0;
                __syncthreads();
                for (unsigned e0 = 0; e0 < cnt; e0 += MG_THREADS) {
                    const unsigned e = e0 + threadIdx.x;
                    const unsigned int b = e < cnt ? __float_as_uint(cand[e]) : 0u;
                    hist_add(hist, e < cnt && (b & lowmask) == lowfix, (b >> sh) & (unsigned)(nbin - 1));
                }
                __syncthreads();
                block_find_bin(hist, nbin, krank, false, wsum, res);
                lowfix |= res[0] << sh; lowmask |= (unsigned)(nbin - 1) << sh; krank -= res[1];
                __syncthreads();
                rem = sh;
            }
            v1b |= lowfix;
        }
        const float v1 = __uint_as_float(v1b);
        if (npos & 1u) med = v1;
        else {
            unsigned int le = 0, mn2 = 0x7f800000u;
            if (!resolved)
                for (unsigned e = threadIdx.x; e < cnt; e += MG_THREADS) { const unsigned int b = __float_as_uint(cand[e]); if (b <= v1b) ++le; else mn2 = min(mn2, b); }
            #pragma unroll
            for (int o = 16; o > 0; o >>= 1) { le += __shfl_xor_sync(FULLMASK, le, o); mn2 = min(mn2, __shfl_xor_sync(FULLMASK, mn2, o)); }
            if (threadIdx.x == 0) { res[0] = 0; res[1] = 0x7f800000u; }
            __syncthreads();
            if (lane == 0) { if (le) atomicAdd(&res[0], le); atomicMin(&res[1], mn2); }
            __syncthreads();
            const unsigned int le_all = resolved ? cnt : res[0];
            const unsigned int v2b = (le_all >= kin + 2) ? v1b : (res[1] != 0x7f800000u ? res[1] : s_min);
            med = v1 * 0.5f + __uint_as_float(v2b) * 0.5f;       // Statistics.middle(a, b) = a/2 + b/2
        }
    }
    if (threadIdx.x == 0) med_out[g] = med;
    // zy[row][0..M) = masked z row, zy[row][M..2M) = masked y row
    float* og = zy + (int64_t)g * d.B * d.c * d.M2;
    #pragma unroll 4
    for (int v = threadIdx.x; v < V2; v += MG_THREADS) {
        const bool isz = v < VZ;
        const float4 f4 = isz ? zg4[v] : yg4[v - VZ];
        const float fv[4] = {f4.x, f4.y, f4.z, f4.w};
        const int e0 = 4 * (isz ? v : v - VZ);
        int np = e0 / d.M, m = e0 - np * d.M;
        if ((d.M & 1) == 0) {
            // M even: e0 and m are even, so each PAIR of values stays inside one row and its destination is 8-byte aligned: two 8-byte stores
            // instead of four 4-byte ones (the scalar stores, with their per-element row arithmetic, were 40 % of this kernel's stall samples)
            float* o0 = og + (int64_t)np * d.M2 + (isz ? 0 : d.M) + m;
            *reinterpret_cast<float2*>(o0) = make_float2(fv[0] >= med ? d.mf * fv[0] : 0.f, fv[1] >= med ? d.mf * fv[1] : 0.f);
            m += 2; if (m == d.M) { m = 0; ++np; }
            float* o1 = og + (int64_t)np * d.M2 + (isz ? 0 : d.M) + m;
            *reinterpret_cast<float2*>(o1) = make_float2(fv[2] >= med ? d.mf * fv[2] : 0.f, fv[3] >= med ? d.mf * fv[3] : 0.f);
        } else {
            #pragma unroll
            for (int i = 0; i < 4; ++i) {
                og[(int64_t)np * d.M2 + (isz ? 0 : d.M) + m] = fv[i] >= med ? d.mf * fv[i] : 0.f;
                if (++m == d.M) { m = 0; ++np; }
            }
        }
    }
    for (int e = 4 * V2 + threadIdx.x; e < E2; e += MG_THREADS) {
        const int ee = e < EZ ? e : e - EZ;
        const int np = ee / d.M, m = ee - np * d.M;
        const float f = e < EZ ? zg[e] : yg[e - EZ];
        og[(int64_t)np * d.M2 + (e < EZ ? 0 : d.M) + m] = f >= med ? d.mf * f : 0.f;
    }
}

// U2 "corr2d" for many groups, fp32: out[n,i,k] (+)= sum_{a<h} sum_{j<2M} A[n,i+a,j] F[a][j][k]   (model.jl:214,251)
// One CTA per sequence.  The sequence's rows (c x 2M, row stride 2M+1 so that the row tiles of a warp fall into different banks)
// stay in shared memory; F is streamed one window offset at a time (2M x K floats, double-buffered through registers).
// Register tiles of 4 rows x 8 filters: per (a, j) a thread issues 4 broadcast row loads + 2 LDS.128 for 32 FMAs.
#define C2B_THREADS 256          // upper bound; launched with the number of register tiles rounded up to a warp (>= 64), so that one round covers the sequence
#define C2B_PRE 10               // float4 of the next F slice a thread holds (600 float4 over >= 64 threads)
template <int KK>
__global__ void __launch_bounds__(C2B_THREADS) k_corr2d_b(const float* __restrict__ A, const float* __restrict__ filt, int64_t filt_gs,
                                                          float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float rb_smem[];
    constexpr int KT = KK / 8;                                  // filter tiles of 8
    const int rt_n = (d.l + 3) >> 2;                            // row tiles of 4
    const int rows_pad = rt_n * 4 + d.h - 1;                    // rows a tile may touch
    const int ldA = d.M2 + 1;
    float* sA = rb_smem;                                        // [rows_pad][ldA]
    float* sF = sA + ((rows_pad * ldA + 3) & ~3);               // [2][2M*KK]
    const int64_t n = blockIdx.x;
    const float* F = filt + (n / d.B) * filt_gs;
    const float* a_src = A + n * d.c * d.M2;
    const int fsz = d.M2 * KK, fv = fsz >> 2;                   // floats / float4 per window offset
    for (int e = threadIdx.x; e < rows_pad * d.M2; e += blockDim.x) {
        const int r = e / d.M2, j = e - r * d.M2;
        sA[r * ldA + j] = r < d.c ? a_src[e] : 0.f;
    }
    const int ntile = rt_n * KT;
    for (int t0 = 0; t0 < ntile; t0 += blockDim.x) {
        const int tile = t0 + threadIdx.x;
        const bool live = tile < ntile;
        const int rt = live ? tile / KT : 0, kt = live ? tile - rt * KT : 0;
        float acc[4][8];
        #pragma unroll
        for (int r = 0; r < 4; ++r)
            #pragma unroll
            for (int k = 0; k < 8; ++k) acc[r][k] = 0.f;
        __syncthreads();                                        // sA filled / previous round done with sF
        for (int v = threadIdx.x; v < fv; v += blockDim.x) reinterpret_cast<float4*>(sF)[v] = reinterpret_cast<const float4*>(F)[v];
        __syncthreads();
        for (int a = 0; a < d.h; ++a) {
            float4 pre[C2B_PRE];                                      // next offset's F slice (2M*KK/4 = 600 float4 over 128 threads)
            const bool more = a + 1 < d.h;
            if (more) {
                const float4* src = reinterpret_cast<const float4*>(F + (int64_t)(a + 1) * fsz);
                #pragma unroll
                for (int u = 0; u < C2B_PRE; ++u) { const int v = threadIdx.x + u * blockDim.x; if (v < fv) pre[u] = src[v]; }
            }
            if (live) {
                const float* f0 = sF + (a & 1) * fsz + kt * 8;
                const float* a0 = sA + (rt * 4 + a) * ldA;
                #pragma unroll 4
                for (int j = 0; j < d.M2; ++j) {
                    const float4 fa = *reinterpret_cast<const float4*>(f0 + j * KK);
                    const float4 fb = *reinterpret_cast<const float4*>(f0 + j * KK + 4);
                    #pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const float av = a0[r * ldA + j];
                        acc[r][0] += av * fa.x; acc[r][1] += av * fa.y; acc[r][2] += av * fa.z; acc[r][3] += av * fa.w;
                        acc[r][4] += av * fb.x; acc[r][5] += av * fb.y; acc[r][6] += av * fb.z; acc[r][7] += av * fb.w;
                    }
                }
            }
            if (more) {
                float4* dst = reinterpret_cast<float4*>(sF + ((a + 1) & 1) * fsz);
                #pragma unroll
                for (int u = 0; u < C2B_PRE; ++u) { const int v = threadIdx.x + u * blockDim.x; if (v < fv) dst[v] = pre[u]; }
            }
            __syncthreads();
        }
        if (live) {
            #pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = rt * 4 + r;
                if (i >= d.l) continue;
                float4* o = reinterpret_cast<float4*>(out + (n * d.l + i) * KK + kt * 8);
                float4 v0 = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]), v1 = make_float4(acc[r][4], acc[r][5], acc[r][6], acc[r][7]);
                if (accumulate) { const float4 p0 = o[0], p1 = o[1]; v0.x += p0.x; v0.y += p0.y; v0.z += p0.z; v0.w += p0.w; v1.x += p1.x; v1.y += p1.y; v1.z += p1.z; v1.w += p1.w; }
                o[0] = v0; o[1] = v1;
            }
        }
    }
}
static inline size_t corr2d_b_smem(const CscDims& d, int KK) {
    const size_t rows_pad = (size_t)(((d.l + 3) >> 2) * 4 + d.h - 1);
    return (((rows_pad * (d.M2 + 1) + 3) & ~(size_t)3) + 2 * (size_t)d.M2 * KK) * 4;
}

// U2 "corr2d" for many groups, register-window form (same contraction as k_corr2d_b, which stays for the shapes this one does not fit).
// k_corr2d_b issues 6 shared-memory loads per 32 FMAs (18 % of the fp32 peak at 64 groups x 200 bp: the load pipe, not the FMA pipe, paces it).
// Here ALL of F (h x 2M x 24 floats = 115 KB) and the CTA's sequences (transposed: [column][row], odd row stride) stay in shared memory, and a
// thread owns TR output rows x 8 filters of one sequence for a RANGE of columns j: per column it loads the TR + h - 1 rows its window touches
// once and slides the h taps over them in registers -- 17 (TR = 6) row loads + 24 16-byte filter loads (the same address across a warp except
// for the three filter tiles: multicast) per 576 FMAs.  Threads = (column range) x (sequence, row tile, filter tile): the column range is
// warp-uniform, its partial sums are combined through shared memory in a fixed order.  The host picks TR, the sequences per CTA and the number
// of column ranges so that the (sequence, row tile, filter tile) combinations fill whole warps (corr2d_s_pick).
#define C2S_MAX_THREADS 384
__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
template <int TR, int H>
__global__ void __launch_bounds__(C2S_MAX_THREADS) k_corr2d_s(const float* __restrict__ A, const float* __restrict__ filt, int64_t filt_gs,
                                                              float* __restrict__ out, int accumulate, int spc, int js_n, int ldr, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float cs_smem[];
    constexpr int KK = 24, WN = TR + H - 1;
    float* sF = cs_smem;                                        // [H][2M][24], later the partial sums [js_n][spc][l][24]
    float* sA = sF + H * d.M2 * KK;                             // [spc][2M][ldr]
    const int64_t n0 = (int64_t)blockIdx.x * spc;
    const float* F = filt + (n0 / d.B) * filt_gs;
    for (int v = threadIdx.x; v < H * d.M2 * KK / 4; v += blockDim.x) cp_async16(sF + 4 * v, F + 4 * v);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int rt_n = (d.l + TR - 1) / TR;
    const int rows_pad = rt_n * TR + H - 1;                     // rows a window may touch (<= ldr); rows >= c read as zero
    // the rows are transposed on the way in by 4-byte asynchronous copies (no register staging: a thread issues all of its ~50 copies back to
    // back and waits once; a load + store loop paid an L2 round trip per few elements and was 40 % of the kernel)
    for (int s = 0; s < spc; ++s) {
        const float* a_src = A + (n0 + s) * d.c * d.M2;
        float* dst = sA + (size_t)s * d.M2 * ldr;
        int r = threadIdx.x / d.M2, j = threadIdx.x - r * d.M2;
        const int dr = blockDim.x / d.M2, dj = blockDim.x - dr * d.M2;
        for (int e = threadIdx.x; e < rows_pad * d.M2; e += blockDim.x) {
            if (r < d.c) cp_async4(dst + j * ldr + r, a_src + e); else dst[j * ldr + r] = 0.f;
            r += dr; j += dj; if (j >= d.M2) { j -= d.M2; ++r; }
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    const int combos = spc * rt_n * 3;
    const int lanes_pad = (combos + 31) & ~31;
    const int js = threadIdx.x / lanes_pad;                     // warp-uniform
    const int cb = threadIdx.x - js * lanes_pad;
    const bool live = cb < combos && js < js_n;
    const int kt = cb % 3, t2 = cb / 3, rt = t2 % rt_n, sq = t2 / rt_n;
    float acc[TR][8];
    #pragma unroll
    for (int r = 0; r < TR; ++r)
        #pragma unroll
        for (int k = 0; k < 8; ++k) acc[r][k] = 0.f;
    if (live) {
        const int j0 = js * d.M2 / js_n, j1 = (js + 1) * d.M2 / js_n;
        const float* ap = sA + (size_t)sq * d.M2 * ldr + rt * TR;
        const float* fp = sF + kt * 8;
        for (int j = j0; j < j1; ++j) {
            float w[WN];
            #pragma unroll
            for (int i = 0; i < WN; ++i) w[i] = ap[j * ldr + i];
            float4 fa = *reinterpret_cast<const float4*>(fp + j * KK), fb = *reinterpret_cast<const float4*>(fp + j * KK + 4);
            #pragma unroll
            for (int a = 0; a < H; ++a) {
                const float4 fa_n = a + 1 < H ? *reinterpret_cast<const float4*>(fp + ((a + 1) * d.M2 + j) * KK) : fa;      // next tap's filters in flight
                const float4 fb_n = a + 1 < H ? *reinterpret_cast<const float4*>(fp + ((a + 1) * d.M2 + j) * KK + 4) : fb;  // under this tap's FMAs
                #pragma unroll
                for (int r = 0; r < TR; ++r) {
                    const float av = w[a + r];
                    acc[r][0] += av * fa.x; acc[r][1] += av * fa.y; acc[r][2] += av * fa.z; acc[r][3] += av * fa.w;
                    acc[r][4] += av * fb.x; acc[r][5] += av * fb.y; acc[r][6] += av * fb.z; acc[r][7] += av * fb.w;
                }
                fa = fa_n; fb = fb_n;
            }
        }
    }
    __syncthreads();                                            // F is no longer read: its space takes the partial sums
    float* part = sF;
    if (live) {
        #pragma unroll
        for (int r = 0; r < TR; ++r) {
            const int i = rt * TR + r;
            if (i < d.l) {
                float4* o = reinterpret_cast<float4*>(part + (((size_t)js * spc + sq) * d.l + i) * KK + kt * 8);
                o[0] = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]); o[1] = make_float4(acc[r][4], acc[r][5], acc[r][6], acc[r][7]);
            }
        }
    }
    __syncthreads();
    const int nout = spc * d.l * KK / 4;                        // the CTA's sequences are consecutive in out
    float4* og = reinterpret_cast<float4*>(out + n0 * d.l * KK);
    const float4* p4 = reinterpret_cast<const float4*>(part);
    for (int v = threadIdx.x; v < nout; v += blockDim.x) {
        float4 sum = p4[v];
        for (int q = 1; q < js_n; ++q) { const float4 t = p4[(size_t)q * nout + v]; sum.x += t.x; sum.y += t.y; sum.z += t.z; sum.w += t.w; }
        if (accumulate) { const float4 t = og[v]; sum.x += t.x; sum.y += t.y; sum.z += t.z; sum.w += t.w; }
        og[v] = sum;
    }
}
struct C2sCfg { int tr = 0, spc = 0, js = 0, ldr = 0, threads = 0; size_t smem = 0; };
// TR in {6, 8}, sequences per CTA in the divisors of the batch, column ranges so that the CTA has ~256-384 threads; tr = 0: the shape does not fit
static inline C2sCfg corr2d_s_pick(const CscDims& d, size_t smem_optin) {
    C2sCfg best; double best_score = 0.0;
    if (d.K != 24 || d.h != 12 || (d.l * 24) % 4) return best;
    for (int tr = 6; tr <= 8; tr += 2)
        for (int spc = 1; spc <= d.B; ++spc) {
            if (d.B % spc) continue;
            const int rt_n = (d.l + tr - 1) / tr, combos = spc * rt_n * 3, lanes_pad = (combos + 31) & ~31;
            if (lanes_pad > C2S_MAX_THREADS) continue;
            int ldr = rt_n * tr + d.h - 1; if (!(ldr & 1)) ++ldr;
            const size_t smem = ((size_t)d.h * d.M2 * 24 + (size_t)spc * d.M2 * ldr) * 4;
            if (smem > smem_optin) continue;
            int js = C2S_MAX_THREADS / lanes_pad;
            while (js > 1 && ((size_t)js * spc * d.l > (size_t)d.h * d.M2 || js > d.M2 / 8)) --js;
            if ((size_t)js * spc * d.l > (size_t)d.h * d.M2) continue;
            const int threads = js * lanes_pad;
            const double score = (double)combos / lanes_pad * std::min(1.0, threads / 256.0) * (tr == 8 ? 1.02 : 1.0);      // a tie goes to the larger tile
            if (score > best_score) { best_score = score; best.tr = tr; best.spc = spc; best.js = js; best.ldr = ldr; best.threads = threads; best.smem = smem; }
        }
    return best;
}

// T3 "dgrad" for many-group launches: of[g][tau][m] (+)= sum_{n in g} sum_p ca[n,p,m] r[n,4p+tau] + cb[n,p,m] r[n,4p+31-tau]
// (model.jl:270-290), one 4-CTA CLUSTER per group.  The per-tau kernels (k_dgrad_c / k_dgrad_b) re-read the codes once per lag: 32 x 30 MB of
// traffic per launch at 64 groups x 200 bp (441 us).  Here a thread owns a tile of 4 lags x 2 filters, the sequence's signal (with the one-hot
// input folded in) is staged in shared memory and the codes are read 8 times (once per lag group, through L1) instead of 32.  CTA s of the
// cluster takes rows [s c/4, (s+1) c/4) of every sequence, its two thread halves alternate halves of those; the partial tiles are added in a
// fixed order (halves, then cluster ranks through distributed shared memory).  f_len = 32, M even and <= 64.
#define DG_THREADS 512
#define DG_SLICES 4                 // measured: 8 slices are slower (121 vs 76 us at 64 groups x 200 bp)
__global__ void __cluster_dims__(1, DG_SLICES, 1) __launch_bounds__(DG_THREADS) k_dgrad_g(const float* __restrict__ ca, const float* __restrict__ cb,
                                                         const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                                         float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float dg_r[];                  // [L4] signal of the current sequence
    __shared__ float s_red[32 * 64];                               // the upper half's tile sums, then this CTA's tile sums
    cg::cluster_group cluster = cg::this_cluster();
    const int g = blockIdx.x, sl = blockIdx.y;
    const int half = threadIdx.x >> 8, t = threadIdx.x & 255;
    const int mpairs = d.M >> 1;
    const bool active = t < 8 * mpairs;
    const int tg = active ? t / mpairs : 0, mp = active ? t - tg * mpairs : 0;
    const int per = (d.c + DG_SLICES - 1) / DG_SLICES;
    const int s_lo = min(d.c, sl * per), s_hi = min(d.c, s_lo + per), p_mid = (s_lo + s_hi + 1) >> 1;
    const int p_lo = half ? p_mid : s_lo, p_hi = half ? s_hi : p_mid;
    float acc[4][2];
    #pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.f;
    for (int nl = 0; nl < d.B; ++nl) {
        const int64_t n = (int64_t)g * d.B + nl;
        __syncthreads();
        for (int q = 4 * s_lo + threadIdx.x; q < min(d.L4, 4 * s_hi + 32); q += DG_THREADS) dg_r[q] = sig_at(sig, bases, sgn, n, q, d);
        __syncthreads();
        if (active) {
            const float* za = ca + (n * d.c) * d.M + 2 * mp;
            const float* yb = cb + (n * d.c) * d.M + 2 * mp;
            for (int p0 = p_lo; p0 < p_hi; p0 += 8) {               // eight rows of codes in flight per thread
                float2 z2[8], y2[8];
                #pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int p = min(p0 + u, p_hi - 1);
                    z2[u] = *reinterpret_cast<const float2*>(za + (int64_t)p * d.M); y2[u] = *reinterpret_cast<const float2*>(yb + (int64_t)p * d.M);
                }
                #pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int p = p0 + u;
                    if (p < p_hi) {
                        const float4 rf = *reinterpret_cast<const float4*>(dg_r + 4 * p + 4 * tg), rr = *reinterpret_cast<const float4*>(dg_r + 4 * p + 28 - 4 * tg);
                        const float f[4] = {rf.x, rf.y, rf.z, rf.w}, rv[4] = {rr.w, rr.z, rr.y, rr.x};
                        #pragma unroll
                        for (int i = 0; i < 4; ++i) { acc[i][0] += z2[u].x * f[i] + y2[u].x * rv[i]; acc[i][1] += z2[u].y * f[i] + y2[u].y * rv[i]; }
                    }
                }
            }
        }
    }
    if (active && half) {
        #pragma unroll
        for (int i = 0; i < 4; ++i) { s_red[(4 * tg + i) * 64 + 2 * mp] = acc[i][0]; s_red[(4 * tg + i) * 64 + 2 * mp + 1] = acc[i][1]; }
    }
    __syncthreads();
    if (active && !half) {
        #pragma unroll
        for (int i = 0; i < 4; ++i) { s_red[(4 * tg + i) * 64 + 2 * mp] += acc[i][0]; s_red[(4 * tg + i) * 64 + 2 * mp + 1] += acc[i][1]; }
    }
    cluster.sync();                                               // every CTA's tile sums are in its s_red
    if (sl == 0 && active && !half) {
        #pragma unroll
        for (int i = 0; i < 4; ++i)
            #pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int tau = 4 * tg + i, m = 2 * mp + u;
                float v = 0.f;
                #pragma unroll
                for (int r = 0; r < DG_SLICES; ++r) v += cluster.map_shared_rank(s_red, r)[tau * 64 + m];
                float* o = of + (int64_t)g * out_gs + tau * d.M + m;
                if (out_gs == 0 && d.G > 1) atomicAdd(o, v);
                else if (accumulate) *o += v; else *o = v;
            }
    }
    cluster.sync();                                               // remote reads of s_red are done
}

// k_dgrad_g with the slice's codes of ALL B sequences and their signals staged in shared memory by asynchronous copies issued up front (one
// wait), then the same tiles and the same order of additions from shared memory: k_dgrad_g walks ~30 dependent rounds of global loads per
// thread (8 rows per round, a signal refill and two block barriers per sequence) and is pure latency (76 us at 64 groups x 200 bp for 30 MB
// of codes and 0.5 GFLOP).  Used when B x (2 x rows x M + 4 x rows + 32) floats fit the opt-in shared memory.
#define DGS_SLICES 4                // CTAs per group of k_dgrad_s (8, i.e. three 60 KB CTAs per SM at 200 bp, measured no faster: 50 vs 47 us)
static inline size_t dgrad_s_smem(const CscDims& d) {
    const size_t per = (size_t)(d.c + DGS_SLICES - 1) / DGS_SLICES;
    return (size_t)d.B * (2 * per * d.M + 4 * per + 32) * 4;
}
__global__ void __cluster_dims__(1, DGS_SLICES, 1) __launch_bounds__(DG_THREADS) k_dgrad_s(const float* __restrict__ ca, const float* __restrict__ cb,
                                                         const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                                         float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    extern __shared__ __align__(16) float dg_sm[];                 // z [B][per][M] | y [B][per][M] | r [B][4 per + 32]
    __shared__ float s_red[32 * 64];                               // the upper half's tile sums, then this CTA's tile sums
    cg::cluster_group cluster = cg::this_cluster();
    const int g = blockIdx.x, sl = blockIdx.y;
    const int half = threadIdx.x >> 8, t = threadIdx.x & 255;
    const int mpairs = d.M >> 1;
    const bool active = t < 8 * mpairs;
    const int tg = active ? t / mpairs : 0, mp = active ? t - tg * mpairs : 0;
    const int per = (d.c + DGS_SLICES - 1) / DGS_SLICES;
    const int s_lo = min(d.c, sl * per), s_hi = min(d.c, s_lo + per), p_mid = (s_lo + s_hi + 1) >> 1;
    const int p_lo = half ? p_mid : s_lo, p_hi = half ? s_hi : p_mid;
    const int rows = s_hi - s_lo, RL = 4 * per + 32;
    float* zs = dg_sm; float* ys = zs + d.B * per * d.M; float* rs = ys + d.B * per * d.M;
    const bool al8 = (((uintptr_t)ca | (uintptr_t)cb) & 7) == 0;
    for (int nl = 0; nl < d.B; ++nl) {
        const int64_t n = (int64_t)g * d.B + nl;
        const float* za = ca + (n * d.c + s_lo) * d.M;
        const float* yb = cb + (n * d.c + s_lo) * d.M;
        float* zd = zs + nl * per * d.M; float* yd = ys + nl * per * d.M;
        if (al8) for (int e = 2 * threadIdx.x; e < rows * d.M; e += 2 * DG_THREADS) { cp_async8(zd + e, za + e); cp_async8(yd + e, yb + e); }
        else for (int e = threadIdx.x; e < rows * d.M; e += DG_THREADS) { zd[e] = za[e]; yd[e] = yb[e]; }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int nl = 0; nl < d.B; ++nl) {
        const int64_t n = (int64_t)g * d.B + nl;
        for (int q = threadIdx.x; q < 4 * rows + 32; q += DG_THREADS) rs[nl * RL + q] = 4 * s_lo + q < d.L4 ? sig_at(sig, bases, sgn, n, 4 * s_lo + q, d) : 0.f;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    float acc[4][2];
    #pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.f;
    if (active) {
        for (int nl = 0; nl < d.B; ++nl) {
            const float* zr = zs + (nl * per - s_lo) * d.M + 2 * mp;
            const float* yr = ys + (nl * per - s_lo) * d.M + 2 * mp;
            const float* rr0 = rs + nl * RL - 4 * s_lo;
            #pragma unroll 4
            for (int p = p_lo; p < p_hi; ++p) {
                const float2 z2 = *reinterpret_cast<const float2*>(zr + p * d.M), y2 = *reinterpret_cast<const float2*>(yr + p * d.M);
                const float4 rf = *reinterpret_cast<const float4*>(rr0 + 4 * p + 4 * tg), rr = *reinterpret_cast<const float4*>(rr0 + 4 * p + 28 - 4 * tg);
                const float f[4] = {rf.x, rf.y, rf.z, rf.w}, rv[4] = {rr.w, rr.z, rr.y, rr.x};
                #pragma unroll
                for (int i = 0; i < 4; ++i) { acc[i][0] += z2.x * f[i] + y2.x * rv[i]; acc[i][1] += z2.y * f[i] + y2.y * rv[i]; }
            }
        }
    }
    if (active && half) {
        #pragma unroll
        for (int i = 0; i < 4; ++i) { s_red[(4 * tg + i) * 64 + 2 * mp] = acc[i][0]; s_red[(4 * tg + i) * 64 + 2 * mp + 1] = acc[i][1]; }
    }
    __syncthreads();
    if (active && !half) {
        #pragma unroll
        for (int i = 0; i < 4; ++i) { s_red[(4 * tg + i) * 64 + 2 * mp] += acc[i][0]; s_red[(4 * tg + i) * 64 + 2 * mp + 1] += acc[i][1]; }
    }
    cluster.sync();                                               // every CTA's tile sums are in its s_red
    if (sl == 0 && active && !half) {
        #pragma unroll
        for (int i = 0; i < 4; ++i)
            #pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int tau = 4 * tg + i, m = 2 * mp + u;
                float v = 0.f;
                #pragma unroll
                for (int r = 0; r < DGS_SLICES; ++r) v += cluster.map_shared_rank(s_red, r)[tau * 64 + m];
                float* o = of + (int64_t)g * out_gs + tau * d.M + m;
                if (out_gs == 0 && d.G > 1) atomicAdd(o, v);
                else if (accumulate) *o += v; else *o = v;
            }
    }
    cluster.sync();                                               // remote reads of s_red are done
}

// U3 "fgrad" for many-group launches: of[g][a][j][k] (+)= sum over the group's list entries (n, i, k, v) of v * A[n][i + a][j]  (model.jl:292-302).
// Rows i .. i+h-1 of A are ONE contiguous window of h*2M floats, so filter k's gradient is a sum of ~B*q/K windows.  k_fgrad_l runs one block
// per (k, a, group) -- 18 432 blocks of 128 threads at 64 groups, each repeating the gather and storing 4 bytes every 96 (57 us for 15 MFLOP).
// Here one CTA per (group, 8 filters): warp w gathers filter k0 + w's entries in (sequence, list) order (the order k_fgrad_l adds them in), a
// thread owns window offsets e = tid, tid + 256, ... for all eight filters (coalesced window reads), and stores 32 contiguous bytes per offset.
#define FG_THREADS 256
#define FG_QCAP 96                  // entries kept per filter and group (B * LIST_CAP = 384 slots over 24 filters: 16 expected)
__global__ void __launch_bounds__(FG_THREADS) k_fgrad_g(const float* __restrict__ A, const float* __restrict__ x, const int32_t* __restrict__ lcnt,
                                                        const uint16_t* __restrict__ lidx, const float* __restrict__ lval,
                                                        float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    __shared__ int s_off[8][FG_QCAP];             // window start (floats) of the entry
    __shared__ float s_v[8][FG_QCAP];
    __shared__ int s_cnt[8];
    __shared__ int s_dense;
    const int g = blockIdx.x, k0 = blockIdx.y * 8;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int HJ = d.h * d.M2;
    if (threadIdx.x == 0) s_dense = 0;
    __syncthreads();
    {   // warp w: ordered gather of the entries with fil == k0 + w
        const int total_slots = d.B * LIST_CAP;
        int running = 0;
        for (int base0 = 0; base0 < total_slots; base0 += 32) {
            const int slot = base0 + lane;
            const int b = slot / LIST_CAP, q = slot - b * LIST_CAP;
            bool hit = false; int e = 0; float v = 0.f;
            const int n = g * d.B + b;
            if (slot < total_slots) {
                const int c = lcnt[n];
                if (c > LIST_CAP) s_dense = 1;
                else if (q < c) { e = lidx[(int64_t)n * LIST_CAP + q]; hit = (e % d.K) == k0 + w; if (hit) v = lval[(int64_t)n * LIST_CAP + q]; }
            }
            const unsigned mk = __ballot_sync(FULLMASK, hit);
            if (hit) {
                const int o = running + __popc(mk & ((1u << lane) - 1u));
                if (o < FG_QCAP) { s_off[w][o] = (b * d.c + e / d.K) * d.M2; s_v[w][o] = v; }
            }
            running += __popc(mk);
        }
        if (lane == 0) { s_cnt[w] = running; if (running > FG_QCAP) s_dense = 1; }
    }
    __syncthreads();
    const float* Ag = A + (int64_t)g * d.B * d.c * d.M2;
    const int e = blockIdx.z * FG_THREADS + threadIdx.x;       // this thread's window offset
    const bool live = e < HJ;
    float acc[8];
    #pragma unroll
    for (int kl = 0; kl < 8; ++kl) acc[kl] = 0.f;
    if (!s_dense) {
        #pragma unroll
        for (int kl = 0; kl < 8; ++kl) {
            const int cnt = s_cnt[kl];
            for (int q0 = 0; q0 < cnt; q0 += 8) {           // eight window reads in flight, added in list order
                float wv[8];
                #pragma unroll
                for (int u = 0; u < 8; ++u) wv[u] = (live && q0 + u < cnt) ? Ag[s_off[kl][q0 + u] + e] : 0.f;
                #pragma unroll
                for (int u = 0; u < 8; ++u) if (q0 + u < cnt) acc[kl] += s_v[kl][q0 + u] * wv[u];
            }
        }
    } else {                                      // a list overflowed: walk x itself in the same (sequence, position) order
        #pragma unroll
        for (int kl = 0; kl < 8; ++kl)
            for (int b = 0; b < d.B; ++b)
                for (int i = 0; i < d.l; ++i) {
                    const float xv = x[(((int64_t)g * d.B + b) * d.l + i) * d.K + k0 + kl];
                    if (xv == 0.f) continue;
                    if (live) acc[kl] += xv * Ag[(b * d.c + i) * d.M2 + e];
                }
    }
    if (live) {
        float* op = of + (int64_t)g * out_gs + (int64_t)e * d.K + k0;
        if (out_gs == 0 && d.G > 1) {
            #pragma unroll
            for (int kl = 0; kl < 8; ++kl) atomicAdd(op + kl, acc[kl]);
        } else {
            float4 v0 = make_float4(acc[0], acc[1], acc[2], acc[3]), v1 = make_float4(acc[4], acc[5], acc[6], acc[7]);
            float4* o4 = reinterpret_cast<float4*>(op);
            if (accumulate) { const float4 p0 = o4[0], p1 = o4[1]; v0.x += p0.x; v0.y += p0.y; v0.z += p0.z; v0.w += p0.w; v1.x += p1.x; v1.y += p1.y; v1.z += p1.z; v1.w += p1.w; }
            o4[0] = v0; o4[1] = v1;
        }
    }
}

// U2 "corr2d" restricted to the entries a top-q kept: out[n,i,k] (+)= sum_{a<h} sum_{j<2M} A[n,i+a,j] F[a][j][k] for (i,k) with bits[n][i*K+k] != 0.
// Every corr2d of the reverse pass produces the adjoint of a top-q OUTPUT, and the top-q adjoint (model.jl:190) discards it outside the kept
// support: ~32 dot products of h*2M terms per sequence instead of l*K (x 136 less work at Lb = 200).  One CTA per sequence, one warp per entry.
#define CK_THREADS 256
__global__ void __launch_bounds__(CK_THREADS) k_corr2d_kept(const float* __restrict__ A, const float* __restrict__ filt, int64_t filt_gs, const uint8_t* __restrict__ bits,
                                                            float* __restrict__ out, int accumulate, int transposed, CscDims d) { PDL_SYNC();
    extern __shared__ int ck_list[];                               // [l*K] kept entries (any order: every entry is written by exactly one warp)
    __shared__ int s_cnt;
    const int64_t n = blockIdx.x;
    const int E = d.l * d.K, HJ = d.h * d.M2;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const uint8_t* b = bits + n * E;
    for (int e = threadIdx.x; e < E; e += CK_THREADS) if (b[e]) ck_list[atomicAdd(&s_cnt, 1)] = e;
    __syncthreads();
    const int cnt = s_cnt, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* F = filt + (n / d.B) * filt_gs;
    for (int q = warp; q < cnt; q += CK_THREADS / 32) {
        const int e = ck_list[q], i = e / d.K, k = e - i * d.K;
        const float* rows = A + (n * d.c + i) * d.M2;              // rows i .. i+h-1 are contiguous
        float acc = 0.f;
        if (transposed) {                                          // filt = Ft [K][h*2M] (k_transpose_F): both operands coalesced
            const float* fk = F + (int64_t)k * HJ;
            #pragma unroll 4
            for (int t = lane; t < HJ; t += 32) acc += rows[t] * fk[t];
        } else {
            #pragma unroll 4
            for (int t = lane; t < HJ; t += 32) acc += rows[t] * F[(int64_t)t * d.K + k];
        }
        acc = warp_sum(acc);
        if (lane == 0) { float* o = out + n * E + e; if (accumulate) *o += acc; else *o = acc; }
    }
}


// adjoint of the warm-up wrt D (k_warm_zy_bwd) for many-group launches: one CTA per sequence.  Chunks of 32 positions: all threads load
// z, y, dz, dy of the chunk (every element once, all loads in flight) and leave gz, gy in shared memory; then one thread per (filter position j,
// filter m) adds its four nucleotide rows over the chunk in registers (fixed order).  ONE atomic per (sequence, entry) at the end -- the
// per-element kernel issues 16 float atomics per code entry onto 1600 addresses (0.5 ms at 64 groups x 200 bp).
#define WZ_ROWS 32
__global__ void __launch_bounds__(512) k_warm_zy_bwd_s(const uint8_t* __restrict__ bases, const float* __restrict__ sc, int i_eta,
                                                        const float* __restrict__ z, const float* __restrict__ y,
                                                        const float* __restrict__ dz, const float* __restrict__ dy, float* __restrict__ dD, CscDims d) { PDL_SYNC();
    __shared__ float s_gz[WZ_ROWS * 64], s_gy[WZ_ROWS * 64];
    const int64_t n = blockIdx.x;
    const int t = threadIdx.x;
    const bool active = t < d.fl * d.M;
    const int j = active ? t / d.M : 0, m = active ? t - j * d.M : 0;
    const float eta = sc[i_eta];
    const uint8_t* s = bases + n * d.Lb;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int p0 = 0; p0 < d.c; p0 += WZ_ROWS) {
        const int rows = min(WZ_ROWS, d.c - p0);
        __syncthreads();
        for (int e = t; e < rows * d.M; e += 512) {
            const int64_t o = (n * d.c + p0) * d.M + e;
            const int pl = e / d.M, mm = e - pl * d.M;
            s_gz[pl * 64 + mm] = z[o] > 0.f ? eta * dz[o] : 0.f;
            s_gy[pl * 64 + mm] = y[o] > 0.f ? eta * dy[o] : 0.f;
        }
        __syncthreads();
        if (active)
            for (int pl = 0; pl < rows; ++pl) {
                const int p = p0 + pl;
                const float gz = s_gz[pl * 64 + m], gy = s_gy[pl * 64 + m];
                const int bz = s[p + j], by = 3 - (int)s[p + d.fl - 1 - j];          // z reads D[4j + b], y reads D[4(fl-1-j') + 3 - b] with j' = fl-1-j
                a0 += (bz == 0 ? gz : 0.f) + (by == 0 ? gy : 0.f); a1 += (bz == 1 ? gz : 0.f) + (by == 1 ? gy : 0.f);
                a2 += (bz == 2 ? gz : 0.f) + (by == 2 ? gy : 0.f); a3 += (bz == 3 ? gz : 0.f) + (by == 3 ? gy : 0.f);
            }
    }
    if (!active) return;
    float* o = dD + n * (int64_t)d.f_len * d.M;                    // this sequence's own slice, summed over sequences in order (k_sum_slices)
    o[(4 * j + 0) * d.M + m] = a0; o[(4 * j + 1) * d.M + m] = a1; o[(4 * j + 2) * d.M + m] = a2; o[(4 * j + 3) * d.M + m] = a3;
}
