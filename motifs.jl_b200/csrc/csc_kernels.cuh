// Device kernels of the unrolled convolutional-sparse-coding network in "position space"
// (SURVEY.md Appendix B).  Reference: src/model.jl (all), restated index by index:
//   * z_mask_n zeroes every row of Z,Y that is not a multiple of 4 (model.jl:54-55,176-177,244), so the
//     network lives on c = Lb-7 positions; mapclarge / mapdrange / upsample_nearest / groups=M*B convs
//     (model.jl:46-51,240-241,270-273,285) are indexing, not arithmetic.
//   * the D layer is three bilinear forms (code x filter -> signal, signal x filter -> code,
//     code x signal -> filter) and the F layer three more (x (*) F -> fx, A (x) F -> x, A (x) x -> F);
//     each form's adjoints are the other two, so six kernels serve forward and backward.
// Layouts (fp32): z,y,alpha,beta [NS][c][M]; zy,fx,theta,d,e [NS][c][2M]; x,g [NS][l][K];
//   signals [NS][4Lb]; D [32][M]; F [h][2M][K]; NS = groups * batch, group g owns sequences g*B..g*B+B-1.
// A filter operand is either shared by all groups (gstride 0) or per group (gstride = its size).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct CscDims {
    int B, G, NS, Lb, L4, c, l, M, M2, K, h, q, fl, f_len, npx, npd;
    float mf;
};

#define FULLMASK 0xffffffffu
// Programmatic dependent launch (optional, MB200_PDL=1): every kernel of the step waits for the full completion (and memory
// flush) of its predecessor before touching memory.  A no-op for a kernel launched without the attribute.
#define PDL_SYNC() asm volatile("griddepcontrol.wait;" ::: "memory")
__device__ __forceinline__ float warp_sum(float v) {
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLMASK, v, o);
    return v;
}
// t = q * div + r.  The element-wise kernels index [NS][c][M] tensors with a 64-bit t; a 64-bit division is ~100 instructions and made those
// kernels ALU-bound at a third of the HBM rate, so indices below 2^31 (every shape in practice) take the 32-bit path.
__device__ __forceinline__ void idx_split(int64_t t, int div, int64_t& q, int& r) {
    if (t < 0x80000000LL) { const unsigned tt = (unsigned)t, qq = tt / (unsigned)div; q = qq; r = (int)(tt - qq * (unsigned)div); }
    else { q = t / div; r = (int)(t - q * div); }
}
// block-wide sum (blockDim.x multiple of 32, <= 1024); result valid in thread 0
__device__ __forceinline__ float block_sum(float v) {
    __shared__ float s_part[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) s_part[w] = v;
    __syncthreads();
    float r = 0.f;
    if (w == 0) { r = lane < (int)(blockDim.x >> 5) ? s_part[lane] : 0.f; r = warp_sum(r); }
    return r;
}

// =============================================================================================
// D layer
// =============================================================================================
// A3 warm-up (model.jl:171-179) fused: z = relu(eta*(sum_j D[4j+s[p+j]][m]) - lam*eta), y with the
// reverse-complement filter D[4(fl-1-j) + 3 - s[p+j]][m].  One thread per (n,p,m).
__global__ void __launch_bounds__(256) k_warm_zy(const uint8_t* __restrict__ bases, const float* __restrict__ D,
                                                 const float* __restrict__ sc, int i_eta, int i_lam,
                                                 float* __restrict__ z, float* __restrict__ y, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M) return;
    int m; int64_t np; idx_split(t, d.M, np, m);
    const int p = (int)(np % d.c);
    const int64_t n = np / d.c;
    const uint8_t* s = bases + n * d.Lb + p;
    float uf = 0.f, ur = 0.f;
    for (int j = 0; j < d.fl; ++j) {
        const int b = s[j];
        uf += D[(4 * j + b) * d.M + m];
        ur += D[(4 * (d.fl - 1 - j) + 3 - b) * d.M + m];
    }
    const float eta = sc[i_eta], lam = sc[i_lam];
    z[t] = fmaxf(eta * uf - lam * eta, 0.f);
    y[t] = fmaxf(eta * ur - lam * eta, 0.f);
}
// adjoint wrt D only (the warm-up scalars are not trainable: model.jl:68,72-73,137)
__global__ void __launch_bounds__(256) k_warm_zy_bwd(const uint8_t* __restrict__ bases, const float* __restrict__ sc, int i_eta,
                                                     const float* __restrict__ z, const float* __restrict__ y,
                                                     const float* __restrict__ dz, const float* __restrict__ dy,
                                                     float* __restrict__ dD, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M) return;
    int m; int64_t np; idx_split(t, d.M, np, m);
    const int p = (int)(np % d.c);
    const int64_t n = np / d.c;
    const float eta = sc[i_eta];
    const float gz = z[t] > 0.f ? eta * dz[t] : 0.f;
    const float gy = y[t] > 0.f ? eta * dy[t] : 0.f;
    if (gz == 0.f && gy == 0.f) return;
    const uint8_t* s = bases + n * d.Lb + p;
    for (int j = 0; j < d.fl; ++j) {
        const int b = s[j];
        if (gz != 0.f) atomicAdd(&dD[(4 * j + b) * d.M + m], gz);
        if (gy != 0.f) atomicAdd(&dD[(4 * (d.fl - 1 - j) + 3 - b) * d.M + m], gy);
    }
}

// T1 "recon": out[n][t] (+)= sum_m sum_{p: 0<=t-4p<f_len} ca[n,p,m] F[t-4p][m] + cb[n,p,m] F[f_len-1-(t-4p)][m]
// (model.jl:238-239, 276-277, 313-314).  One warp per (n,t), lanes over m.
__global__ void __launch_bounds__(256) k_recon(const float* __restrict__ ca, const float* __restrict__ cb,
                                               const float* __restrict__ filt, int64_t filt_gs,
                                               float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= (int64_t)d.NS * d.L4) return;
    const int t = (int)(wid % d.L4);
    const int64_t n = wid / d.L4;
    const float* F = filt + (n / d.B) * filt_gs;
    const int p_hi = min(d.c - 1, t >> 2);
    const int p_lo = max(0, (t - d.f_len + 4) >> 2);            // smallest p with t-4p <= f_len-1
    float acc = 0.f;
    if (p_hi - p_lo < 8) {                                       // f_len = 32: at most 8 positions reach t; unrolled so every load is in flight
        #pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
            const int p = p_lo + pp;
            if (p <= p_hi) {
                const int k = t - 4 * p;
                const float* a = ca + (n * d.c + p) * d.M;
                const float* b = cb + (n * d.c + p) * d.M;
                const float* f0 = F + k * d.M;
                const float* f1 = F + (d.f_len - 1 - k) * d.M;
                for (int m = lane; m < d.M; m += 32) acc += a[m] * f0[m] + b[m] * f1[m];
            }
        }
    } else {
        for (int p = p_lo; p <= p_hi; ++p) {
            const int k = t - 4 * p;
            const float* a = ca + (n * d.c + p) * d.M;
            const float* b = cb + (n * d.c + p) * d.M;
            const float* f0 = F + k * d.M;
            const float* f1 = F + (d.f_len - 1 - k) * d.M;
            for (int m = lane; m < d.M; m += 32) acc += a[m] * f0[m] + b[m] * f1[m];
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) { if (accumulate) out[wid] += acc; else out[wid] = acc; }
}

// signal element with the one-hot input folded in: sig[n][t] + sgn * S[n][t], S[n][4p+a] = (base[n][p]==a)
__device__ __forceinline__ float sig_at(const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn, int64_t n, int t, const CscDims& d) {
    float v = sig[n * d.L4 + t];
    if (sgn != 0.f && bases[n * d.Lb + (t >> 2)] == (t & 3)) v += sgn;
    return v;
}

// T2 "corr_sig": oa[n,p,m] (+)= sum_k r[n,4p+k] F[k][m];  ob[n,p,m] (+)= sum_k r[n,4p+k] F[f_len-1-k][m],  r = sig + sgn*S
// (model.jl:240-241 z_grad/y_grad data terms).  One thread per (n,p,m).
__global__ void __launch_bounds__(256) k_corr_sig(const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                                  const float* __restrict__ filt, int64_t filt_gs,
                                                  float* __restrict__ oa, float* __restrict__ ob, int accumulate, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M) return;
    int m; int64_t np; idx_split(t, d.M, np, m);
    const int p = (int)(np % d.c);
    const int64_t n = np / d.c;
    const float* F = filt + (n / d.B) * filt_gs;
    float a = 0.f, b = 0.f;
    #pragma unroll 8
    for (int k = 0; k < d.f_len; ++k) {
        const float r = sig_at(sig, bases, sgn, n, 4 * p + k, d);
        a += r * F[k * d.M + m];
        b += r * F[(d.f_len - 1 - k) * d.M + m];
    }
    if (accumulate) { oa[t] += a; ob[t] += b; } else { oa[t] = a; ob[t] = b; }
}

// T3 "dgrad": of[g][tau][m] (+)= sum_{n in g} sum_p ca[n,p,m] r[n,4p+tau] + cb[n,p,m] r[n,4p+f_len-1-tau]
// (model.jl:270-290 conv_code_diff + mapdrange, with r = sumZD+sumYRD+S there).  grid.y = group; one thread per
// (tau,m).  When the output is shared by all groups (out_gs == 0) contributions are added atomically.
__global__ void __launch_bounds__(256) k_dgrad(const float* __restrict__ ca, const float* __restrict__ cb,
                                               const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                               float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.f_len * d.M) return;
    const int g = blockIdx.y;
    const int m = t % d.M, tau = t / d.M;
    float acc = 0.f;
    for (int64_t n = (int64_t)g * d.B; n < (int64_t)(g + 1) * d.B; ++n)
        for (int p = 0; p < d.c; ++p) {
            const float a = ca[(n * d.c + p) * d.M + m], b = cb[(n * d.c + p) * d.M + m];
            if (a != 0.f) acc += a * sig_at(sig, bases, sgn, n, 4 * p + tau, d);
            if (b != 0.f) acc += b * sig_at(sig, bases, sgn, n, 4 * p + d.f_len - 1 - tau, d);
        }
    float* o = of + (int64_t)g * out_gs + t;
    if (out_gs == 0 && d.G > 1) atomicAdd(o, acc);
    else if (accumulate) *o += acc; else *o = acc;
}

// =============================================================================================
// F layer
// =============================================================================================
// U2 "corr2d": out[n,i,k] (+)= sum_{a<h} sum_{j<2M} A[n,i+a,j] F[a][j][k]   (model.jl:214,251). One thread per (n,i,k).
__global__ void __launch_bounds__(128) k_corr2d(const float* __restrict__ A, const float* __restrict__ filt, int64_t filt_gs,
                                                float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.l * d.K) return;
    const int k = (int)(t % d.K);
    const int64_t ni = t / d.K;
    const int i = (int)(ni % d.l);
    const int64_t n = ni / d.l;
    const float* F = filt + (n / d.B) * filt_gs + k;
    const float* a0 = A + (n * d.c + i) * d.M2;
    float acc = 0.f;
    const int hj = d.h * d.M2;                      // rows i..i+h-1 of A are contiguous: A[n,i+a,j] = a0[a*2M + j]
    for (int e = 0; e < hj; ++e) {
        const float av = a0[e];
        if (av != 0.f) acc += av * F[(int64_t)e * d.K];
    }
    if (accumulate) out[t] += acc; else out[t] = acc;
}

// U1 "tconv": out[n,i,j] (+)= sum_a sum_k x[n,i-a,k] F[a][j][k], 0 <= i-a < l   (model.jl:229,263,294,316,370).
// One thread per (n,i,j); x holds few non-zeros (top-q), so zero rows are skipped (warp-uniform test).
__global__ void __launch_bounds__(128) k_tconv(const float* __restrict__ x, const float* __restrict__ filt, int64_t filt_gs,
                                               float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M2) return;
    const int j = (int)(t % d.M2);
    const int64_t ni = t / d.M2;
    const int i = (int)(ni % d.c);
    const int64_t n = ni / d.c;
    const float* F = filt + (n / d.B) * filt_gs;
    float acc = 0.f;
    const int a_lo = max(0, i - d.l + 1), a_hi = min(d.h - 1, i);
    for (int a = a_lo; a <= a_hi; ++a) {
        const float* xr = x + (n * d.l + (i - a)) * d.K;
        const float* fr = F + ((int64_t)a * d.M2 + j) * d.K;
        for (int k = 0; k < d.K; ++k) {
            const float xv = xr[k];
            if (xv != 0.f) acc += xv * fr[k];
        }
    }
    if (accumulate) out[t] += acc; else out[t] = acc;
}

// U3 "fgrad": of[g][a][j][k] (+)= sum_{n in g} sum_{i<l} A[n,a+i,j] x[n,i,k]   (model.jl:292-302). grid.y = group.
__global__ void __launch_bounds__(128) k_fgrad(const float* __restrict__ A, const float* __restrict__ x,
                                               float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.h * d.M2 * d.K) return;
    const int g = blockIdx.y;
    const int k = t % d.K;
    const int aj = t / d.K;
    const int j = aj % d.M2, a = aj / d.M2;
    float acc = 0.f;
    for (int64_t n = (int64_t)g * d.B; n < (int64_t)(g + 1) * d.B; ++n) {
        const float* Ar = A + (n * d.c + a) * d.M2 + j;
        const float* xr = x + n * d.l * d.K + k;
        for (int i = 0; i < d.l; ++i) {
            const float xv = xr[(int64_t)i * d.K];
            if (xv != 0.f) acc += xv * Ar[(int64_t)i * d.M2];
        }
    }
    float* o = of + (int64_t)g * out_gs + t;
    if (out_gs == 0 && d.G > 1) atomicAdd(o, acc);
    else if (accumulate) *o += acc; else *o = acc;
}

// =============================================================================================
// element-wise updates (with their adjoints)
// =============================================================================================
// A8 (model.jl:240-244): zn = relu(z - eta*(gz + rho*(z - fx[:, :M] - alpha)) - lam*eta), same for y with fx[:, M:], beta.
__global__ void __launch_bounds__(256) k_zy_update(const float* __restrict__ z, const float* __restrict__ y,
                                                   const float* __restrict__ gz, const float* __restrict__ gy,
                                                   const float* __restrict__ fx, const float* __restrict__ al, const float* __restrict__ be,
                                                   const float* __restrict__ sc, int i_eta, int i_lam, int i_rho,
                                                   float* __restrict__ zn, float* __restrict__ yn, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M) return;
    int m; int64_t np; idx_split(t, d.M, np, m);
    const float eta = sc[i_eta], lam = sc[i_lam], rho = sc[i_rho];
    const float l = fx[np * d.M2 + m], r = fx[np * d.M2 + d.M + m];
    zn[t] = fmaxf(z[t] - eta * (gz[t] + rho * (z[t] - l - al[t])) - lam * eta, 0.f);
    yn[t] = fmaxf(y[t] - eta * (gy[t] + rho * (y[t] - r - be[t])) - lam * eta, 0.f);
}
__global__ void __launch_bounds__(256) k_zy_update_bwd(const float* __restrict__ z, const float* __restrict__ y,
                                                       const float* __restrict__ gz, const float* __restrict__ gy,
                                                       const float* __restrict__ fx, const float* __restrict__ al, const float* __restrict__ be,
                                                       const float* __restrict__ sc, int i_eta, int i_lam, int i_rho,
                                                       const float* __restrict__ zn, const float* __restrict__ yn,
                                                       const float* __restrict__ dzn, const float* __restrict__ dyn,
                                                       float* __restrict__ dz, float* __restrict__ dy, float* __restrict__ dgz, float* __restrict__ dgy,
                                                       float* __restrict__ dfx, float* __restrict__ dal, float* __restrict__ dbe,
                                                       float* __restrict__ part, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float s_eta = 0.f, s_lam = 0.f, s_rho = 0.f;
    if (t < (int64_t)d.NS * d.c * d.M) {
        int m; int64_t np; idx_split(t, d.M, np, m);
        const float eta = sc[i_eta], lam = sc[i_lam], rho = sc[i_rho];
        const float tz = zn[t] > 0.f ? dzn[t] : 0.f;
        const float ty = yn[t] > 0.f ? dyn[t] : 0.f;
        const float l = fx[np * d.M2 + m], r = fx[np * d.M2 + d.M + m];
        const float ez = z[t] - l - al[t], ey = y[t] - r - be[t];
        dz[t] += tz * (1.f - eta * rho);
        dy[t] += ty * (1.f - eta * rho);
        dgz[t] += -eta * tz;
        dgy[t] += -eta * ty;
        dfx[np * d.M2 + m] += eta * rho * tz;
        dfx[np * d.M2 + d.M + m] += eta * rho * ty;
        dal[t] += eta * rho * tz;
        dbe[t] += eta * rho * ty;
        s_eta = tz * (-(gz[t] + rho * ez) - lam) + ty * (-(gy[t] + rho * ey) - lam);
        s_lam = -eta * (tz + ty);
        s_rho = -eta * (tz * ez + ty * ey);
    }
    s_eta = block_sum(s_eta); s_lam = block_sum(s_lam); s_rho = block_sum(s_rho);
    if (threadIdx.x == 0) { part[3 * blockIdx.x] = s_eta; part[3 * blockIdx.x + 1] = s_lam; part[3 * blockIdx.x + 2] = s_rho; }      // block partials, summed in block order (k_sum_slots)
}

// A4 (model.jl:194-210): zy' = mf * [zy >= median{zy > 0 over the whole batch}] * zy.  One block per group:
// exact selection of the middle order statistic(s) of the positive entries by an MSB-first radix select on the
// float bit patterns (positive floats order like unsigned ints), then the mask is applied.  med[g] is kept for
// the adjoint (the mask is a constant for AD: model.jl:208).
__device__ __forceinline__ float zy_elem(const float* __restrict__ z, const float* __restrict__ y, int64_t e, const CscDims& d) {
    // e indexes [n_local][p][j] inside the group's block of B*c*2M values
    const int j = (int)(e % d.M2);
    const int64_t np = e / d.M2;
    return j < d.M ? z[np * d.M + j] : y[np * d.M + (j - d.M)];
}
__global__ void __launch_bounds__(1024) k_mask_scale(const float* __restrict__ z, const float* __restrict__ y,
                                                     float* __restrict__ zy, float* __restrict__ med_out, CscDims d) { PDL_SYNC();
    __shared__ unsigned int hist[256];
    __shared__ unsigned int s_prefix, s_rank, s_cnt;
    __shared__ float s_med;
    const int g = blockIdx.x;
    const int64_t E = (int64_t)d.B * d.c * d.M2;
    const float* zg = z + (int64_t)g * d.B * d.c * d.M;
    const float* yg = y + (int64_t)g * d.B * d.c * d.M;
    // 1. number of positive entries
    unsigned int cnt = 0;
    for (int64_t e = threadIdx.x; e < E; e += blockDim.x) cnt += zy_elem(zg, yg, e, d) > 0.f;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if (cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    const unsigned int npos = s_cnt;
    float med = -INFINITY;                                       // no positives: "no mask" (model.jl:197-198,209)
    if (npos > 0) {
        // ranks (0-based, ascending) of the middle element(s): odd -> npos/2 ; even -> npos/2-1 and npos/2
        const unsigned int k1 = (npos & 1u) ? npos / 2 : npos / 2 - 1;
        if (threadIdx.x == 0) { s_prefix = 0; s_rank = k1; }
        for (int shift = 24; shift >= 0; shift -= 8) {
            if (threadIdx.x < 256) hist[threadIdx.x] = 0;
            __syncthreads();
            const unsigned int prefix = s_prefix;
            const unsigned int pmask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
            for (int64_t e = threadIdx.x; e < E; e += blockDim.x) {
                const float v = zy_elem(zg, yg, e, d);
                if (v > 0.f) {
                    const unsigned int b = __float_as_uint(v);
                    if ((b & pmask) == prefix) atomicAdd(&hist[(b >> shift) & 255u], 1u);
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                unsigned int r = s_rank, c0 = 0; int bin = 0;
                for (; bin < 256; ++bin) { if (c0 + hist[bin] > r) break; c0 += hist[bin]; }
                s_rank = r - c0; s_prefix = prefix | ((unsigned int)bin << shift);
            }
            __syncthreads();
        }
        const float v1 = __uint_as_float(s_prefix);
        if (npos & 1u) med = v1;
        else {
            // next order statistic: v1 again if it is repeated past rank k1, else the smallest value above v1
            __syncthreads();
            if (threadIdx.x == 0) { s_cnt = 0; s_prefix = 0x7f800000u; }
            __syncthreads();
            unsigned int le = 0, mn = 0x7f800000u;
            for (int64_t e = threadIdx.x; e < E; e += blockDim.x) {
                const float v = zy_elem(zg, yg, e, d);
                if (v > 0.f) { if (v <= v1) ++le; else mn = min(mn, __float_as_uint(v)); }
            }
            if (le) atomicAdd(&s_cnt, le);
            atomicMin(&s_prefix, mn);
            __syncthreads();
            const float v2 = (s_cnt >= k1 + 2) ? v1 : __uint_as_float(s_prefix);
            med = v1 * 0.5f + v2 * 0.5f;                         // Statistics.middle(a, b) = a/2 + b/2
        }
    }
    if (threadIdx.x == 0) { s_med = med; med_out[g] = med; }
    __syncthreads();
    med = s_med;
    float* og = zy + (int64_t)g * E;
    for (int64_t e = threadIdx.x; e < E; e += blockDim.x) {
        const float v = zy_elem(zg, yg, e, d);
        og[e] = v >= med ? d.mf * v : 0.f;
    }
}
__global__ void __launch_bounds__(256) k_mask_scale_bwd(const float* __restrict__ z, const float* __restrict__ y, const float* __restrict__ med,
                                                        const float* __restrict__ dzy, float* __restrict__ dz, float* __restrict__ dy, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M2) return;
    int j; int64_t np; idx_split(t, d.M2, np, j);
    int64_t gq; int gr; idx_split(np, d.c * d.B, gq, gr);
    const float mg = med[gq];
    if (j < d.M) { const int64_t o = np * d.M + j; if (z[o] >= mg) dz[o] += d.mf * dzy[t]; }
    else { const int64_t o = np * d.M + (j - d.M); if (y[o] >= mg) dy[o] += d.mf * dzy[t]; }
}

// A9 input: dd = fx - (zy' - [alpha beta])   (model.jl:248-250)
__global__ void __launch_bounds__(256) k_d_build(const float* __restrict__ fx, const float* __restrict__ zy, const float* __restrict__ al,
                                                 const float* __restrict__ be, float* __restrict__ dd, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M2) return;
    int j; int64_t np; idx_split(t, d.M2, np, j);
    const float ab = j < d.M ? al[np * d.M + j] : be[np * d.M + j - d.M];
    dd[t] = fx[t] - (zy[t] - ab);
}
__global__ void __launch_bounds__(256) k_d_build_bwd(const float* __restrict__ ddd, float* __restrict__ dfx, float* __restrict__ dzy,
                                                     float* __restrict__ dal, float* __restrict__ dbe, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M2) return;
    int j; int64_t np; idx_split(t, d.M2, np, j);
    const float g = ddd[t];
    dfx[t] += g; dzy[t] -= g;
    if (j < d.M) dal[np * d.M + j] += g; else dbe[np * d.M + j - d.M] += g;
}

// A5/A6/A9 (model.jl:181-192, 212-216, 252-253): v = (xprev ? xprev : 0) - sgn_omega*omega*g ; keep entries >= the
// q-th largest of the sequence.  One block per sequence; MSB-first radix select on order-preserving keys.
__device__ __forceinline__ unsigned int fkey(float v) { unsigned int b = __float_as_uint(v); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float fkey_inv(unsigned int k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
__global__ void __launch_bounds__(256) k_topq(const float* __restrict__ xprev, const float* __restrict__ g, const float* __restrict__ sc, int i_om,
                                              float coef, float* __restrict__ xout, uint8_t* __restrict__ bit, float* __restrict__ vq_out, CscDims d) { PDL_SYNC();
    __shared__ unsigned int hist[256];
    __shared__ unsigned int s_prefix, s_rank;
    const int64_t n = blockIdx.x;
    const int E = d.l * d.K;
    const float om = coef * sc[i_om];
    const float* gp = g + n * E;
    const float* xp = xprev ? xprev + n * E : nullptr;
    if (threadIdx.x == 0) { s_prefix = 0; s_rank = (unsigned int)(E - d.q); }      // q-th largest = ascending rank E-q
    for (int shift = 24; shift >= 0; shift -= 8) {
        hist[threadIdx.x] = 0;
        __syncthreads();
        const unsigned int prefix = s_prefix;
        const unsigned int pmask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
        for (int e = threadIdx.x; e < E; e += blockDim.x) {
            const float v = (xp ? xp[e] : 0.f) + om * gp[e];
            const unsigned int kk = fkey(v);
            if ((kk & pmask) == prefix) atomicAdd(&hist[(kk >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int r = s_rank, c0 = 0; int bin = 0;
            for (; bin < 256; ++bin) { if (c0 + hist[bin] > r) break; c0 += hist[bin]; }
            s_rank = r - c0; s_prefix = prefix | ((unsigned int)bin << shift);
        }
        __syncthreads();
    }
    const float vq = fkey_inv(s_prefix);
    if (threadIdx.x == 0) vq_out[n] = vq;
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
        const float v = (xp ? xp[e] : 0.f) + om * gp[e];
        const bool keep = v >= vq;
        xout[n * E + e] = keep ? v : 0.f;
        bit[n * E + e] = keep;
    }
}
__global__ void __launch_bounds__(256) k_topq_bwd(const uint8_t* __restrict__ bit, const float* __restrict__ g, const float* __restrict__ sc, int i_om,
                                                  float coef, const float* __restrict__ dxout, float* __restrict__ dxprev, float* __restrict__ dg,
                                                  float* __restrict__ dsc, int om_trainable, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float s = 0.f;
    if (t < (int64_t)d.NS * d.l * d.K) {
        const float gr = bit[t] ? dxout[t] : 0.f;
        if (dxprev) dxprev[t] += gr;
        dg[t] += coef * sc[i_om] * gr;
        s = coef * gr * g[t];
    }
    if (om_trainable) { s = block_sum(s); if (threadIdx.x == 0 && s != 0.f) atomicAdd(&dsc[i_om], s); }
}

// dual update (model.jl:265-266): an = al + fx[:, :M] - z ; bn = be + fx[:, M:] - y
__global__ void __launch_bounds__(256) k_dual(const float* __restrict__ al, const float* __restrict__ be, const float* __restrict__ fx,
                                              const float* __restrict__ z, const float* __restrict__ y, float* __restrict__ an, float* __restrict__ bn, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M) return;
    int m; int64_t np; idx_split(t, d.M, np, m);
    an[t] = (al ? al[t] : 0.f) + fx[np * d.M2 + m] - z[t];
    bn[t] = (be ? be[t] : 0.f) + fx[np * d.M2 + d.M + m] - y[t];
}
__global__ void __launch_bounds__(256) k_dual_bwd(const float* __restrict__ dan, const float* __restrict__ dbn, float* __restrict__ dal, float* __restrict__ dbe,
                                                  float* __restrict__ dfx, float* __restrict__ dz, float* __restrict__ dy, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.c * d.M) return;
    int m; int64_t np; idx_split(t, d.M, np, m);
    const float ga = dan[t], gb = dbn[t];
    if (dal) { dal[t] += ga; dbe[t] += gb; }
    dfx[np * d.M2 + m] += ga; dfx[np * d.M2 + d.M + m] += gb;
    dz[t] -= ga; dy[t] -= gb;
}

// out = a - b - (c ? c : 0)   over [NS][c][2M]   (e = fx - (zy + theta), model.jl:294; theta' = theta + fx - zy, :370 as out = fx - zy + theta)
__global__ void __launch_bounds__(256) k_sub3(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c3, float csign,
                                              float* __restrict__ out, int64_t n) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    out[t] = a[t] - b[t] + (c3 ? csign * c3[t] : 0.f);
}
__global__ void __launch_bounds__(256) k_sub3_bwd(const float* __restrict__ dout, float* __restrict__ da, float* __restrict__ db, float* __restrict__ dc3,
                                                  float csign, int64_t n) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const float g = dout[t];
    da[t] += g; db[t] -= g;
    if (dc3) dc3[t] += csign * g;
}

// A10 update (model.jl:287-288): Dn[g][4j+a][m] = D exp(-mu G) / sum_a' (D exp(-mu G)).  One thread per (g,j,m).
__global__ void __launch_bounds__(256) k_d_update(const float* __restrict__ D, int64_t D_gs, const float* __restrict__ G, const float* __restrict__ sc, int i_mu,
                                                  float* __restrict__ Dn, CscDims d) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.G * d.fl * d.M) return;
    const int m = t % d.M;
    const int gj = t / d.M;
    const int j = gj % d.fl, g = gj / d.fl;
    const float mu = sc[i_mu];
    const float* Dg = D + (int64_t)g * D_gs;
    const int64_t gs = (int64_t)d.f_len * d.M;
    float u[4], s = 0.f;
    #pragma unroll
    for (int a = 0; a < 4; ++a) { const int o = (4 * j + a) * d.M + m; u[a] = Dg[o] * expf(-mu * G[g * gs + o]); s += u[a]; }
    #pragma unroll
    for (int a = 0; a < 4; ++a) Dn[g * gs + (4 * j + a) * d.M + m] = u[a] / s;
}
__global__ void __launch_bounds__(256) k_d_update_bwd(const float* __restrict__ D, int64_t D_gs, const float* __restrict__ G, const float* __restrict__ sc, int i_mu,
                                                      const float* __restrict__ Dn, const float* __restrict__ dDn,
                                                      float* __restrict__ dD, int64_t dD_gs, float* __restrict__ dG, float* __restrict__ part, CscDims d) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    float s_mu = 0.f;
    if (t < d.G * d.fl * d.M) {
        const int m = t % d.M;
        const int gj = t / d.M;
        const int j = gj % d.fl, g = gj / d.fl;
        const float mu = sc[i_mu];
        const float* Dg = D + (int64_t)g * D_gs;
        const int64_t gs = (int64_t)d.f_len * d.M;
        float u[4], s = 0.f, dot = 0.f;
        #pragma unroll
        for (int a = 0; a < 4; ++a) { const int o = (4 * j + a) * d.M + m; u[a] = Dg[o] * expf(-mu * G[g * gs + o]); s += u[a]; dot += dDn[g * gs + o] * Dn[g * gs + o]; }
        #pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int o = (4 * j + a) * d.M + m;
            const float du = (dDn[g * gs + o] - dot) / s;                 // d loss / d u_a
            const float e = expf(-mu * G[g * gs + o]);
            const float gD = du * e;
            if (dD_gs == 0 && d.G > 1) atomicAdd(&dD[o], gD); else dD[(int64_t)g * dD_gs + o] += gD;
            dG[g * gs + o] += du * u[a] * (-mu);
            s_mu += du * u[a] * (-G[g * gs + o]);
        }
    }
    s_mu = block_sum(s_mu);
    if (threadIdx.x == 0) part[blockIdx.x] = s_mu;
}

// A11 update (model.jl:304-308): Fu = relu(F - kap*Fg - kap*kaps) ; Fn[:,:,k] = Fu[:,:,k] / ||Fu[:,:,k]||_2.  One block per (g,k).
__global__ void __launch_bounds__(256) k_f_update(const float* __restrict__ F, int64_t F_gs, const float* __restrict__ Fg, const float* __restrict__ sc,
                                                  int i_kap, int i_kaps, float* __restrict__ Fn, float* __restrict__ nrm, CscDims d) { PDL_SYNC();
    __shared__ float s_n;
    const int k = blockIdx.x % d.K, g = blockIdx.x / d.K;
    const float kap = sc[i_kap], kaps = sc[i_kaps];
    const int HJ = d.h * d.M2;
    const int64_t gs = (int64_t)HJ * d.K;
    const float* Fp = F + (int64_t)g * F_gs;
    float ss = 0.f;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {
        const float u = fmaxf(Fp[(int64_t)e * d.K + k] - kap * Fg[g * gs + (int64_t)e * d.K + k] - kap * kaps, 0.f);
        ss += u * u;
    }
    ss = block_sum(ss);
    if (threadIdx.x == 0) { s_n = sqrtf(ss); nrm[g * d.K + k] = s_n; }
    __syncthreads();
    const float nn = s_n;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {
        const float u = fmaxf(Fp[(int64_t)e * d.K + k] - kap * Fg[g * gs + (int64_t)e * d.K + k] - kap * kaps, 0.f);
        Fn[g * gs + (int64_t)e * d.K + k] = u / nn;
    }
}
__global__ void __launch_bounds__(256) k_f_update_bwd(const float* __restrict__ Fn, const float* __restrict__ nrm, const float* __restrict__ Fg,
                                                      const float* __restrict__ sc, int i_kap, int i_kaps, const float* __restrict__ dFn,
                                                      float* __restrict__ dF, int64_t dF_gs, float* __restrict__ dFg, float* __restrict__ part, CscDims d) { PDL_SYNC();
    __shared__ float s_dot;
    const int k = blockIdx.x % d.K, g = blockIdx.x / d.K;
    const float kap = sc[i_kap], kaps = sc[i_kaps];
    const int HJ = d.h * d.M2;
    const int64_t gs = (int64_t)HJ * d.K;
    const float nn = nrm[g * d.K + k];
    float dot = 0.f;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) dot += dFn[g * gs + (int64_t)e * d.K + k] * Fn[g * gs + (int64_t)e * d.K + k];
    dot = block_sum(dot);
    if (threadIdx.x == 0) s_dot = dot;
    __syncthreads();
    dot = s_dot;
    float s_kap = 0.f, s_kaps = 0.f;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {
        const int64_t o = g * gs + (int64_t)e * d.K + k;
        const float fn = Fn[o];
        if (fn > 0.f) {                                             // relu active (u = fn * nn > 0)
            const float du = (dFn[o] - dot * fn) / nn;
            if (dF_gs == 0 && d.G > 1) atomicAdd(&dF[(int64_t)e * d.K + k], du); else dF[(int64_t)g * dF_gs + (int64_t)e * d.K + k] += du;
            dFg[o] += -kap * du;
            s_kap += du * (-Fg[o] - kaps);
            s_kaps += du * (-kap);
        }
    }
    s_kap = block_sum(s_kap); s_kaps = block_sum(s_kaps);
    if (threadIdx.x == 0) { part[2 * blockIdx.x] = s_kap; part[2 * blockIdx.x + 1] = s_kaps; }
}

// A12 (model.jl:310-325): loss[g] = (1/B) (sum (recon - S)^2 + sum (fx - zy)^2).  One block per group.
__global__ void __launch_bounds__(1024) k_loss(const float* __restrict__ recon, const uint8_t* __restrict__ bases, const float* __restrict__ fx,
                                               const float* __restrict__ zy, float* __restrict__ loss, CscDims d) { PDL_SYNC();
    const int g = blockIdx.x;
    float a = 0.f, b = 0.f;
    const int64_t n0 = (int64_t)g * d.B;
    for (int64_t e = threadIdx.x; e < (int64_t)d.B * d.L4; e += blockDim.x) {
        const int64_t n = n0 + e / d.L4; const int t = (int)(e % d.L4);
        const float r = sig_at(recon, bases, -1.f, n, t, d);
        a += r * r;
    }
    const int64_t E2 = (int64_t)d.B * d.c * d.M2, o2 = n0 * d.c * d.M2;
    for (int64_t e = threadIdx.x; e < E2; e += blockDim.x) { const float v = fx[o2 + e] - zy[o2 + e]; b += v * v; }
    a = block_sum(a); b = block_sum(b);
    if (threadIdx.x == 0) { loss[g * 3 + 0] = (a + b) / (float)d.B; loss[g * 3 + 1] = a / (float)d.B; loss[g * 3 + 2] = b / (float)d.B; }
}
// seeds the adjoints: d loss_total / d loss[g] = wgt (1/G for the mean over groups)
__global__ void __launch_bounds__(256) k_loss_bwd(const float* __restrict__ recon, const uint8_t* __restrict__ bases, const float* __restrict__ fx,
                                                  const float* __restrict__ zy, float wgt, float* __restrict__ drecon, float* __restrict__ dfx,
                                                  float* __restrict__ dzy, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const float s = 2.f * wgt / (float)d.B;
    if (t < (int64_t)d.NS * d.L4) drecon[t] += s * sig_at(recon, bases, -1.f, t / d.L4, (int)(t % d.L4), d);
    if (t < (int64_t)d.NS * d.c * d.M2) { const float v = s * (fx[t] - zy[t]); dfx[t] += v; dzy[t] -= v; }
}

// =============================================================================================
// parameter preparation (model.jl:139-169) and its adjoint; raw parameter vector in Flux.params order
// =============================================================================================
// scalars: eff = raw^2
// the eight scalar arrays sit in separate places of the raw parameter vector: one launch squares them all (warp w = segment w)
struct ScalarSegs { int raw_off[8], eff_idx[8], n[8], nseg; };
__global__ void __launch_bounds__(256) k_prep_scalars(const float* __restrict__ raw, float* __restrict__ eff, ScalarSegs sg) { PDL_SYNC();
    const int w = threadIdx.x >> 5;
    if (w >= sg.nseg) return;
    for (int i = threadIdx.x & 31; i < sg.n[w]; i += 32) { const float r = raw[sg.raw_off[w] + i]; eff[sg.eff_idx[w] + i] = r * r; }
}
__global__ void __launch_bounds__(256) k_prep_scalars_bwd(const float* __restrict__ raw, const float* __restrict__ deff, float* __restrict__ draw, ScalarSegs sg) { PDL_SYNC();
    const int w = threadIdx.x >> 5;
    if (w >= sg.nseg) return;
    for (int i = threadIdx.x & 31; i < sg.n[w]; i += 32) draw[sg.raw_off[w] + i] += 2.f * raw[sg.raw_off[w] + i] * deff[sg.eff_idx[w] + i];
}
// D: raw is Julia (32,1,M) column-major = raw[m*32 + 4j + a]; eff[(4j+a)*M + m] = (raw^2 + 1e-3) / sum_a'(...)
__global__ void k_prep_D(const float* __restrict__ raw, float* __restrict__ eff, CscDims d) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.fl * d.M) return;
    const int m = t % d.M, j = t / d.M;
    float u[4], s = 0.f;
    #pragma unroll
    for (int a = 0; a < 4; ++a) { const float r = raw[m * d.f_len + 4 * j + a]; u[a] = r * r + 0.001f; s += u[a]; }
    #pragma unroll
    for (int a = 0; a < 4; ++a) eff[(4 * j + a) * d.M + m] = u[a] / s;
}
__global__ void k_prep_D_bwd(const float* __restrict__ raw, const float* __restrict__ eff, const float* __restrict__ deff, float* __restrict__ draw, CscDims d) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= d.fl * d.M) return;
    const int m = t % d.M, j = t / d.M;
    float s = 0.f, dot = 0.f;
    #pragma unroll
    for (int a = 0; a < 4; ++a) { const float r = raw[m * d.f_len + 4 * j + a]; s += r * r + 0.001f; dot += deff[(4 * j + a) * d.M + m] * eff[(4 * j + a) * d.M + m]; }
    #pragma unroll
    for (int a = 0; a < 4; ++a) {
        const float r = raw[m * d.f_len + 4 * j + a];
        draw[m * d.f_len + 4 * j + a] += (deff[(4 * j + a) * d.M + m] - dot) / s * 2.f * r;
    }
}
// F: raw is Julia (h,2M,1,K) column-major = raw[(k*2M + j)*h + a]; eff[(a*2M + j)*K + k] = raw^2 / sqrt(sum_{a,j} raw^4). One block per k.
__global__ void __launch_bounds__(256) k_prep_F(const float* __restrict__ raw, float* __restrict__ eff, float* __restrict__ nrm, CscDims d) { PDL_SYNC();
    __shared__ float s_n;
    const int k = blockIdx.x;
    const int HJ = d.h * d.M2;
    float ss = 0.f;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {           // e = j*h + a in raw order
        const float r = raw[(int64_t)k * HJ + e]; const float u = r * r; ss += u * u;
    }
    ss = block_sum(ss);
    if (threadIdx.x == 0) { s_n = sqrtf(ss); nrm[k] = s_n; }
    __syncthreads();
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {
        const int a = e % d.h, j = e / d.h;
        const float r = raw[(int64_t)k * HJ + e];
        eff[((int64_t)a * d.M2 + j) * d.K + k] = r * r / s_n;
    }
}
__global__ void __launch_bounds__(256) k_prep_F_bwd(const float* __restrict__ raw, const float* __restrict__ eff, const float* __restrict__ nrm,
                                                    const float* __restrict__ deff, float* __restrict__ draw, CscDims d) { PDL_SYNC();
    __shared__ float s_dot;
    const int k = blockIdx.x;
    const int HJ = d.h * d.M2;
    float dot = 0.f;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {
        const int a = e % d.h, j = e / d.h;
        const int64_t o = ((int64_t)a * d.M2 + j) * d.K + k;
        dot += deff[o] * eff[o];
    }
    dot = block_sum(dot);
    if (threadIdx.x == 0) s_dot = dot;
    __syncthreads();
    dot = s_dot;
    const float nn = nrm[k];
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) {
        const int a = e % d.h, j = e / d.h;
        const int64_t o = ((int64_t)a * d.M2 + j) * d.K + k;
        const float r = raw[(int64_t)k * HJ + e];
        draw[(int64_t)k * HJ + e] += (deff[o] - dot * eff[o]) / nn * 2.f * r;     // u = r^2, eff = u/||u||
    }
}

// unpack the selected sequences' bases from the 2-bit store: bases[n][p] for n in idx
__global__ void __launch_bounds__(256) k_unpack_bases(const uint32_t* __restrict__ words, int64_t rowwords, const int64_t* __restrict__ idx,
                                                      uint8_t* __restrict__ bases, CscDims d) { PDL_SYNC();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)d.NS * d.Lb) return;
    const int p = (int)(t % d.Lb);
    const int64_t n = t / d.Lb;
    const uint32_t w = words[idx[n] * rowwords + (p >> 4)];
    bases[t] = (uint8_t)((w >> ((p & 15) * 2)) & 3u);
}

// AdaBelief (Flux 0.14.6 Optimise.AdaBelief, restated; see oracle/csc_oracle.py) over the trainable vector, fp32.
// Deterministic sums of the tape's shared adjoints.  Where many CTAs or groups feed one adjoint, float atomics would add in an order that
// varies from run to run; instead each group, sequence or block writes its own slice or slot, and these kernels add them in a fixed order.
// dst[i] += sum over k < ns of src[k * n + i], k ascending.
__global__ void __launch_bounds__(256) k_sum_slices(const float* __restrict__ src, int ns, int64_t n, float* __restrict__ dst) { PDL_SYNC();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float a = 0.f;
    for (int k = 0; k < ns; ++k) a += src[(int64_t)k * n + i];
    dst[i] += a;
}
struct SlotRange { int32_t idx, n, stride, pad; int64_t off; };   // scalar idx receives src[off + i * stride], i < n
// one block per scalar: its ranges in table order, each summed by a fixed thread assignment and block_sum
__global__ void __launch_bounds__(256) k_sum_slots(const float* __restrict__ src, const SlotRange* __restrict__ r, int nr, float* __restrict__ dsc) { PDL_SYNC();
    float tot = 0.f;
    for (int k = 0; k < nr; ++k) {
        if (r[k].idx != (int)blockIdx.x) continue;
        float a = 0.f;
        for (int i = threadIdx.x; i < r[k].n; i += blockDim.x) a += src[r[k].off + (int64_t)i * r[k].stride];
        tot += block_sum(a);
    }
    if (threadIdx.x == 0) dsc[blockIdx.x] += tot;
}

// err: the fused reverse pass's error word (null for handles without it); a step it flagged is not applied (csc.cu: fused_fallback)
__global__ void __launch_bounds__(256) k_adabelief(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ mt, float* __restrict__ st,
                                                   float eta, float b1, float b2, float eps2, float c1, float c2, int n, const unsigned int* __restrict__ err) { PDL_SYNC();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || (err && *err)) return;
    const float gr = g[t];
    const float m = b1 * mt[t] + (1.f - b1) * gr;
    const float dv = gr - m;
    const float s = b2 * st[t] + (1.f - b2) * dv * dv + eps2;
    mt[t] = m; st[t] = s;
    p[t] -= eta * m / c1 / (sqrtf(s / c2) + eps2);
}
// l1 = sum |prep_syntax_filters(F)| (train.jl:47): per k sum(r^2)/sqrt(sum r^4).  One block per k writes its term to out[k]; the host
// adds the K terms in index order (no atomics: the statistic is bit-identical across data-parallel ranks).
__global__ void __launch_bounds__(256) k_l1_F(const float* __restrict__ raw, float* __restrict__ out, CscDims d, const unsigned int* __restrict__ err) { PDL_SYNC();
    if (err && *err) return;                      // block-uniform: no update was applied (k_adabelief)
    const int k = blockIdx.x;
    const int HJ = d.h * d.M2;
    float s2 = 0.f, s4 = 0.f;
    for (int e = threadIdx.x; e < HJ; e += blockDim.x) { const float r = raw[(int64_t)k * HJ + e]; const float u = r * r; s2 += u; s4 += u * u; }
    s2 = block_sum(s2); s4 = block_sum(s4);
    if (threadIdx.x == 0) out[k] = s2 / sqrtf(s4);
}

// =============================================================================================
// Faster variants used by the tape (the plain kernels above remain as fallbacks for unusual shapes).
// =============================================================================================
#define LIST_CAP 64        // non-zeros kept per sequence in a code list; more -> consumers use their dense path

// warp-parallel search of the radix bin that contains ascending rank `rank` in a 256-bin histogram.
// Call with the 32 lanes of one warp; returns (bin, count below the bin) to every lane.
__device__ __forceinline__ void find_bin(const unsigned int* hist, unsigned int rank, int* bin_out, unsigned int* below_out) {
    const int lane = threadIdx.x & 31;
    unsigned int h[8], s = 0;
    #pragma unroll
    for (int i = 0; i < 8; ++i) { h[i] = hist[lane * 8 + i]; s += h[i]; }
    unsigned int inc = s;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned int y = __shfl_up_sync(FULLMASK, inc, o); if (lane >= o) inc += y; }
    const unsigned int exc = inc - s;
    const unsigned hitmask = __ballot_sync(FULLMASK, inc > rank);
    const int owner = __ffs(hitmask) - 1;                          // first lane whose cumulative count exceeds rank
    int bin = 0; unsigned int below = 0;
    if (lane == owner) {
        unsigned int c0 = exc; int b = 0;
        #pragma unroll
        for (; b < 8; ++b) { if (c0 + h[b] > rank) break; c0 += h[b]; }
        bin = lane * 8 + b; below = c0;
    }
    *bin_out = __shfl_sync(FULLMASK, bin, owner);
    *below_out = __shfl_sync(FULLMASK, below, owner);
}

// histogram increment with intra-warp aggregation: lanes that hit the same bin elect one leader (values of one
// group/sequence share their leading bytes, so plain shared-memory atomics would serialise on one bin)
__device__ __forceinline__ void hist_add(unsigned int* hist, bool active, unsigned int bin) {
    const unsigned act = __ballot_sync(FULLMASK, active);
    if (!active) return;
    const unsigned peers = __match_any_sync(act, bin);
    if ((threadIdx.x & 31) == (__ffs(peers) - 1)) atomicAdd(&hist[bin], (unsigned int)__popc(peers));
}

// U2 dense: one block (4 warps) computes ROWS consecutive output rows (same sequence) for all KK outputs.  The
// 1200-long reduction index e = a*2M + j is strided over the 128 threads; every F row (KK floats) is loaded once per
// ROWS rows; partial sums are combined by warp shuffles and a small shared-memory reduction (fixed order).
template <int KK, int ROWS>
__global__ void __launch_bounds__(128) k_corr2d_w(const float* __restrict__ A, const float* __restrict__ filt, int64_t filt_gs,
                                                  float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    __shared__ float s_part[4][ROWS * KK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tiles = (d.l + ROWS - 1) / ROWS;
    const int64_t n = blockIdx.x / tiles;
    const int i0 = (int)(blockIdx.x % tiles) * ROWS;
    const float* F = filt + (n / d.B) * filt_gs;
    const float* a0 = A + (n * d.c + i0) * d.M2;
    const int hj = d.h * d.M2;
    const int rows = min(ROWS, d.l - i0);
    float acc[ROWS][KK];
    #pragma unroll
    for (int r = 0; r < ROWS; ++r)
        #pragma unroll
        for (int k = 0; k < KK; ++k) acc[r][k] = 0.f;
    #pragma unroll 2
    for (int e = threadIdx.x; e < hj; e += 128) {
        float av[ROWS];
        #pragma unroll
        for (int r = 0; r < ROWS; ++r) av[r] = r < rows ? a0[(int64_t)r * d.M2 + e] : 0.f;
        const float4* fr = reinterpret_cast<const float4*>(F + (int64_t)e * KK);
        #pragma unroll
        for (int k4 = 0; k4 < KK / 4; ++k4) {
            const float4 f = __ldg(fr + k4);
            #pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                acc[r][4 * k4 + 0] += av[r] * f.x; acc[r][4 * k4 + 1] += av[r] * f.y;
                acc[r][4 * k4 + 2] += av[r] * f.z; acc[r][4 * k4 + 3] += av[r] * f.w;
            }
        }
    }
    #pragma unroll
    for (int r = 0; r < ROWS; ++r)
        #pragma unroll
        for (int k = 0; k < KK; ++k) {
            const float v = warp_sum(acc[r][k]);
            if (lane == ((r * KK + k) & 31)) s_part[warp][r * KK + k] = v;
        }
    __syncthreads();
    for (int o = threadIdx.x; o < rows * KK; o += 128) {
        const float v = (s_part[0][o] + s_part[1][o]) + (s_part[2][o] + s_part[3][o]);
        float* op = out + (n * d.l + i0) * KK + o;
        if (accumulate) *op += v; else *op = v;
    }
}

// T3, one block per (group, tau): 16 reduction phases x 64 filter slots, deterministic shared-memory reduction.
__global__ void __launch_bounds__(1024) k_dgrad_b(const float* __restrict__ ca, const float* __restrict__ cb,
                                                  const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                                  float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    __shared__ float s_red[16][64];
    const int tau = blockIdx.x, g = blockIdx.y;
    const int m = threadIdx.x & 63, ph = threadIdx.x >> 6;
    float acc = 0.f;
    if (m < d.M) {
        const int total = d.B * d.c;                               // (n_local, p) pairs of the group
        const int64_t n0 = (int64_t)g * d.B;
        #pragma unroll 4
        for (int e = ph; e < total; e += 16) {
            const int nl = e / d.c, p = e - nl * d.c;
            const int64_t n = n0 + nl;
            const float a = ca[(n * d.c + p) * d.M + m], b = cb[(n * d.c + p) * d.M + m];
            acc += a * sig_at(sig, bases, sgn, n, 4 * p + tau, d) + b * sig_at(sig, bases, sgn, n, 4 * p + d.f_len - 1 - tau, d);
        }
    }
    s_red[ph][m] = acc;
    __syncthreads();
    if (ph == 0 && m < d.M) {
        float v = 0.f;
        #pragma unroll
        for (int i = 0; i < 16; ++i) v += s_red[i][m];
        float* o = of + (int64_t)g * out_gs + tau * d.M + m;
        if (out_gs == 0 && d.G > 1) atomicAdd(o, v);
        else if (accumulate) *o += v; else *o = v;
    }
}

// ordered block-wide compaction helper: returns the exclusive prefix of `cnt` over threads (blockDim.x == 256)
__device__ __forceinline__ int block_excl_scan256(int cnt, int* total) {
    __shared__ int s_w[9];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = cnt;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(FULLMASK, inc, o); if (lane >= o) inc += y; }
    __syncthreads();
    if (lane == 31) s_w[w] = inc;
    __syncthreads();
    if (threadIdx.x == 0) { int run = 0; for (int i = 0; i < 8; ++i) { const int t = s_w[i]; s_w[i] = run; run += t; } s_w[8] = run; }
    __syncthreads();
    *total = s_w[8];
    return s_w[w] + inc - cnt;
}

// A5 top-q with the sequence's values staged in shared memory (E = l*K floats of dynamic smem) and an ordered
// non-zero list (entry = flat index i*K+k, value) written for the sparse consumers.
__global__ void __launch_bounds__(256) k_topq_s(const float* __restrict__ xprev, const float* __restrict__ g, const float* __restrict__ sc, int i_om,
                                                float coef, float* __restrict__ xout, uint8_t* __restrict__ bit,
                                                int32_t* __restrict__ lcnt, uint16_t* __restrict__ lidx, float* __restrict__ lval, CscDims d) { PDL_SYNC();
    extern __shared__ float s_v[];
    __shared__ unsigned int hist[256];
    __shared__ unsigned int s_prefix, s_rank;
    const int64_t n = blockIdx.x;
    const int E = d.l * d.K;
    const float om = coef * sc[i_om];
    for (int e = threadIdx.x; e < E; e += blockDim.x) s_v[e] = (xprev ? xprev[n * E + e] : 0.f) + om * g[n * E + e];
    if (threadIdx.x == 0) { s_prefix = 0; s_rank = (unsigned int)(E - d.q); }
    for (int shift = 24; shift >= 0; shift -= 8) {
        hist[threadIdx.x] = 0;
        __syncthreads();
        const unsigned int prefix = s_prefix;
        const unsigned int pmask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
        for (int e0 = 0; e0 < E; e0 += blockDim.x) {
            const int e = e0 + threadIdx.x;
            const unsigned int kk = e < E ? fkey(s_v[e]) : 0u;
            hist_add(hist, e < E && (kk & pmask) == prefix, (kk >> shift) & 255u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            int bin; unsigned int below;
            find_bin(hist, s_rank, &bin, &below);
            __syncwarp();
            if (threadIdx.x == 0) { s_rank -= below; s_prefix = prefix | ((unsigned int)bin << shift); }
        }
        __syncthreads();
    }
    const float vq = fkey_inv(s_prefix);
    // contiguous chunk per thread so that the list is ordered by flat index
    const int per = (E + 255) / 256;
    const int e0 = threadIdx.x * per, e1 = min(E, e0 + per);
    int cnt = 0;
    for (int e = e0; e < e1; ++e) {
        const float v = s_v[e];
        const bool keep = v >= vq;
        xout[n * E + e] = keep ? v : 0.f;
        bit[n * E + e] = keep;
        cnt += keep && v != 0.f;
    }
    int total;
    int o = block_excl_scan256(cnt, &total);
    for (int e = e0; e < e1; ++e) {
        const float v = s_v[e];
        if (v >= vq && v != 0.f) { if (o < LIST_CAP) { lidx[n * LIST_CAP + o] = (uint16_t)e; lval[n * LIST_CAP + o] = v; } ++o; }
    }
    if (threadIdx.x == 0) lcnt[n] = total;
}
// adjoint of top-q, one block per sequence; also writes the ordered non-zero list of dg (the x-role operand of the
// adjoints of corr2d) and reduces d omega.
__global__ void __launch_bounds__(256) k_topq_s_bwd(const uint8_t* __restrict__ bit, const float* __restrict__ g, const float* __restrict__ sc, int i_om,
                                                    float coef, const float* __restrict__ dxout, float* __restrict__ dxprev, float* __restrict__ dg,
                                                    float* __restrict__ part, int om_trainable,
                                                    int32_t* __restrict__ lcnt, uint16_t* __restrict__ lidx, float* __restrict__ lval, CscDims d) { PDL_SYNC();
    const int64_t n = blockIdx.x;
    const int E = d.l * d.K;
    const float om = coef * sc[i_om];
    const int per = (E + 255) / 256;
    const int e0 = threadIdx.x * per, e1 = min(E, e0 + per);
    float s = 0.f; int cnt = 0;
    for (int e = e0; e < e1; ++e) {
        const int64_t t = n * E + e;
        const float gr = bit[t] ? dxout[t] : 0.f;
        if (dxprev) dxprev[t] += gr;
        const float dgv = om * gr;
        dg[t] = dgv;                       // g has a single consumer (this op): plain store, the arena value is overwritten
        s += coef * gr * g[t];
        cnt += dgv != 0.f;
    }
    int total;
    int o = block_excl_scan256(cnt, &total);
    for (int e = e0; e < e1; ++e) {
        const float dgv = dg[n * E + e];
        if (dgv != 0.f) { if (o < LIST_CAP) { lidx[n * LIST_CAP + o] = (uint16_t)e; lval[n * LIST_CAP + o] = dgv; } ++o; }
    }
    if (threadIdx.x == 0) lcnt[n] = total;
    if (om_trainable) { s = block_sum(s); if (threadIdx.x == 0) part[blockIdx.x] = s; }
}

// U1 with the x operand given as a list: one block per (n, i), threads over j.
__global__ void __launch_bounds__(128) k_tconv_l(const float* __restrict__ x, const int32_t* __restrict__ lcnt, const uint16_t* __restrict__ lidx,
                                                 const float* __restrict__ lval, const float* __restrict__ filt, int64_t filt_gs,
                                                 float* __restrict__ out, int accumulate, CscDims d) { PDL_SYNC();
    __shared__ int s_i[LIST_CAP], s_k[LIST_CAP];
    __shared__ float s_v[LIST_CAP];
    const int64_t n = blockIdx.x / d.c;
    const int i = blockIdx.x % d.c;
    const float* F = filt + (n / d.B) * filt_gs;
    const int cnt = lcnt[n];
    if (cnt <= LIST_CAP) {
        if (threadIdx.x < cnt) {
            const int e = lidx[n * LIST_CAP + threadIdx.x];
            s_i[threadIdx.x] = e / d.K; s_k[threadIdx.x] = e % d.K; s_v[threadIdx.x] = lval[n * LIST_CAP + threadIdx.x];
        }
        __syncthreads();
        for (int j = threadIdx.x; j < d.M2; j += blockDim.x) {
            float acc = 0.f;
            for (int q = 0; q < cnt; ++q) {
                const int a = i - s_i[q];
                if (a >= 0 && a < d.h) acc += s_v[q] * F[((int64_t)a * d.M2 + j) * d.K + s_k[q]];
            }
            float* o = out + (n * d.c + i) * d.M2 + j;
            if (accumulate) *o += acc; else *o = acc;
        }
    } else {                                     // dense path (more than LIST_CAP non-zeros in this sequence)
        const int a_lo = max(0, i - d.l + 1), a_hi = min(d.h - 1, i);
        for (int j = threadIdx.x; j < d.M2; j += blockDim.x) {
            float acc = 0.f;
            for (int a = a_lo; a <= a_hi; ++a) {
                const float* xr = x + (n * d.l + (i - a)) * d.K;
                const float* fr = F + ((int64_t)a * d.M2 + j) * d.K;
                for (int k = 0; k < d.K; ++k) { const float xv = xr[k]; if (xv != 0.f) acc += xv * fr[k]; }
            }
            float* o = out + (n * d.c + i) * d.M2 + j;
            if (accumulate) *o += acc; else *o = acc;
        }
    }
}

// U3 with the x operand given as lists: one block per (k, a, group); the group's entries with fil == k are gathered in
// order (sequence, position) by the first warp and every thread accumulates one j over them.
__global__ void __launch_bounds__(128) k_fgrad_l(const float* __restrict__ A, const float* __restrict__ x, const int32_t* __restrict__ lcnt,
                                                 const uint16_t* __restrict__ lidx, const float* __restrict__ lval,
                                                 float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    __shared__ int s_n[256], s_i[256];
    __shared__ float s_v[256];
    __shared__ int s_cnt, s_dense;
    const int k = blockIdx.x, a = blockIdx.y, g = blockIdx.z;
    // gather: the group's list entries form a virtual array [b][q] (q < LIST_CAP); every thread tests a few of them with
    // independent loads, then an ordered block-wide compaction keeps (sequence, position) order
    __shared__ int s_wsum[8];
    if (threadIdx.x == 0) { s_cnt = 0; s_dense = 0; }
    __syncthreads();
    const int total_slots = d.B * LIST_CAP;
    int running = 0;
    for (int base0 = 0; base0 < total_slots; base0 += blockDim.x) {          // block-uniform trip count (3 for B = 6)
        const int slot = base0 + threadIdx.x;
        const int b = slot / LIST_CAP, q = slot - b * LIST_CAP;
        bool hit = false; int e = 0; float v = 0.f; int64_t n = 0;
        if (slot < total_slots) {
            n = (int64_t)g * d.B + b;
            const int c = lcnt[n];
            if (c > LIST_CAP) s_dense = 1;
            else if (q < c) { e = lidx[n * LIST_CAP + q]; hit = (e % d.K) == k; if (hit) v = lval[n * LIST_CAP + q]; }
        }
        const unsigned mk = __ballot_sync(FULLMASK, hit);
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane == 0) s_wsum[w] = __popc(mk);
        __syncthreads();
        int woff = 0, tot = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { if (i < w) woff += s_wsum[i]; tot += s_wsum[i]; }
        if (hit) {
            const int o = running + woff + __popc(mk & ((1u << lane) - 1u));
            if (o < 256) { s_n[o] = (int)n; s_i[o] = e / d.K; s_v[o] = v; }
        }
        running += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) { s_cnt = running; if (running > 256) s_dense = 1; }
    __syncthreads();
    if (!s_dense) {
        const int cnt = s_cnt;
        for (int j = threadIdx.x; j < d.M2; j += blockDim.x) {
            float acc = 0.f;
            for (int q = 0; q < cnt; ++q) acc += s_v[q] * A[((int64_t)s_n[q] * d.c + a + s_i[q]) * d.M2 + j];
            float* op = of + (int64_t)g * out_gs + ((int64_t)a * d.M2 + j) * d.K + k;
            if (out_gs == 0 && d.G > 1) atomicAdd(op, acc);
            else if (accumulate) *op += acc; else *op = acc;
        }
    } else {
        for (int j = threadIdx.x; j < d.M2; j += blockDim.x) {
            float acc = 0.f;
            for (int64_t n = (int64_t)g * d.B; n < (int64_t)(g + 1) * d.B; ++n)
                for (int i = 0; i < d.l; ++i) {
                    const float xv = x[(n * d.l + i) * d.K + k];
                    if (xv != 0.f) acc += xv * A[(n * d.c + a + i) * d.M2 + j];
                }
            float* op = of + (int64_t)g * out_gs + ((int64_t)a * d.M2 + j) * d.K + k;
            if (out_gs == 0 && d.G > 1) atomicAdd(op, acc);
            else if (accumulate) *op += acc; else *op = acc;
        }
    }
}

// A4 with the positive entries of the group compacted into shared memory (cap floats of dynamic smem); falls back to
// re-reading global memory in every pass when there are more positives than fit.
__global__ void __launch_bounds__(1024) k_mask_scale_s(const float* __restrict__ z, const float* __restrict__ y,
                                                       float* __restrict__ zy, float* __restrict__ med_out, int cap, CscDims d) { PDL_SYNC();
    extern __shared__ float s_pos[];
    __shared__ unsigned int hist[256];
    __shared__ unsigned int s_prefix, s_rank, s_cnt, s_min;
    __shared__ float s_med;
    const int g = blockIdx.x;
    const int64_t EZ = (int64_t)d.B * d.c * d.M;
    const float* zg = z + (int64_t)g * EZ;
    const float* yg = y + (int64_t)g * EZ;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    // 1. compact positives (order is irrelevant for order statistics)
    for (int64_t e0 = 0; e0 < 2 * EZ; e0 += blockDim.x) {
        const int64_t e = e0 + threadIdx.x;
        float v = 0.f;
        if (e < EZ) v = zg[e]; else if (e < 2 * EZ) v = yg[e - EZ];
        const bool pos = v > 0.f;
        const unsigned m = __ballot_sync(FULLMASK, pos);
        unsigned base = 0;
        if (lane == 0 && m) base = atomicAdd(&s_cnt, __popc(m));
        base = __shfl_sync(FULLMASK, base, 0);
        if (pos) { const unsigned o = base + __popc(m & ((1u << lane) - 1u)); if (o < (unsigned)cap) s_pos[o] = v; }
    }
    __syncthreads();
    const unsigned int npos = s_cnt;
    const bool in_smem = npos <= (unsigned)cap;
    float med = -INFINITY;
    if (npos > 0) {
        const unsigned int k1 = (npos & 1u) ? npos / 2 : npos / 2 - 1;
        if (threadIdx.x == 0) { s_prefix = 0; s_rank = k1; }
        for (int shift = 24; shift >= 0; shift -= 8) {
            if (threadIdx.x < 256) hist[threadIdx.x] = 0;
            __syncthreads();
            const unsigned int prefix = s_prefix;
            const unsigned int pmask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
            if (in_smem) {
                for (unsigned e0 = 0; e0 < npos; e0 += blockDim.x) {
                    const unsigned e = e0 + threadIdx.x;
                    const unsigned int b = e < npos ? __float_as_uint(s_pos[e]) : 0u;
                    hist_add(hist, e < npos && (b & pmask) == prefix, (b >> shift) & 255u);
                }
            } else {
                for (int64_t e = threadIdx.x; e < 2 * EZ; e += blockDim.x) {
                    const float v = e < EZ ? zg[e] : yg[e - EZ];
                    if (v > 0.f) { const unsigned int b = __float_as_uint(v); if ((b & pmask) == prefix) atomicAdd(&hist[(b >> shift) & 255u], 1u); }
                }
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                int bin; unsigned int below;
                find_bin(hist, s_rank, &bin, &below);
                __syncwarp();
                if (threadIdx.x == 0) { s_rank -= below; s_prefix = prefix | ((unsigned int)bin << shift); }
            }
            __syncthreads();
        }
        const float v1 = __uint_as_float(s_prefix);
        if (npos & 1u) med = v1;
        else {
            __syncthreads();
            if (threadIdx.x == 0) { s_cnt = 0; s_min = 0x7f800000u; }
            __syncthreads();
            unsigned int le = 0, mn = 0x7f800000u;
            if (in_smem) {
                for (unsigned e = threadIdx.x; e < npos; e += blockDim.x) { const float v = s_pos[e]; if (v <= v1) ++le; else mn = min(mn, __float_as_uint(v)); }
            } else {
                for (int64_t e = threadIdx.x; e < 2 * EZ; e += blockDim.x) {
                    const float v = e < EZ ? zg[e] : yg[e - EZ];
                    if (v > 0.f) { if (v <= v1) ++le; else mn = min(mn, __float_as_uint(v)); }
                }
            }
            if (le) atomicAdd(&s_cnt, le);
            atomicMin(&s_min, mn);
            __syncthreads();
            const float v2 = (s_cnt >= k1 + 2) ? v1 : __uint_as_float(s_min);
            med = v1 * 0.5f + v2 * 0.5f;
        }
    }
    if (threadIdx.x == 0) { s_med = med; med_out[g] = med; }
    __syncthreads();
    med = s_med;
    // 2. apply: rows np = (n_local, p), lanes over m
    const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    float* og = zy + (int64_t)g * d.B * d.c * d.M2;
    for (int np = warp; np < d.B * d.c; np += nw)
        for (int m = lane; m < d.M; m += 32) {
            const float vz = zg[(int64_t)np * d.M + m], vy = yg[(int64_t)np * d.M + m];
            og[(int64_t)np * d.M2 + m] = vz >= med ? d.mf * vz : 0.f;
            og[(int64_t)np * d.M2 + d.M + m] = vy >= med ? d.mf * vy : 0.f;
        }
}

// =============================================================================================
// Thread-block-cluster variants: 8 CTAs cooperate through distributed shared memory (DSMEM), so that a reduction
// that used to run on one SM spreads over 8 while staying ONE launch with a fixed (deterministic) summation order.
// =============================================================================================
#include <cooperative_groups.h>
namespace cg = cooperative_groups;
#define CL 8
#define MS_MAXV 32        // values per thread the cluster median kernel keeps in registers (512 threads: 16384 per CTA)

// T3 on a cluster: CTA r of the cluster reduces slice r of the group's (sequence, position) pairs; the 8 partial rows
// land in CTA 0's shared memory and are summed there in rank order.
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(256) k_dgrad_c(const float* __restrict__ ca, const float* __restrict__ cb,
                                                                            const float* __restrict__ sig, const uint8_t* __restrict__ bases, float sgn,
                                                                            float* __restrict__ of, int64_t out_gs, int accumulate, CscDims d) { PDL_SYNC();
    __shared__ float s_red[4][64];
    __shared__ float s_all[CL][64];
    cg::cluster_group cluster = cg::this_cluster();
    const int r = (int)cluster.block_rank();
    const int tau = blockIdx.x / CL, g = blockIdx.y;
    const int m = threadIdx.x & 63, ph = threadIdx.x >> 6;
    const int total = d.B * d.c;
    const int per = (total + CL - 1) / CL;
    const int e_lo = r * per, e_hi = min(total, e_lo + per);
    float acc = 0.f;
    if (m < d.M) {
        const int64_t n0 = (int64_t)g * d.B;
        #pragma unroll 4
        for (int e = e_lo + ph; e < e_hi; e += 4) {
            const int nl = e / d.c, p = e - nl * d.c;
            const int64_t n = n0 + nl;
            const float a = ca[(n * d.c + p) * d.M + m], b = cb[(n * d.c + p) * d.M + m];
            acc += a * sig_at(sig, bases, sgn, n, 4 * p + tau, d) + b * sig_at(sig, bases, sgn, n, 4 * p + d.f_len - 1 - tau, d);
        }
    }
    s_red[ph][m] = acc;
    __syncthreads();
    if (ph == 0) {
        float* dst = cluster.map_shared_rank(&s_all[0][0], 0);
        dst[r * 64 + m] = (s_red[0][m] + s_red[1][m]) + (s_red[2][m] + s_red[3][m]);
    }
    cluster.sync();
    if (r == 0 && ph == 0 && m < d.M) {
        float v = 0.f;
        #pragma unroll
        for (int i = 0; i < CL; ++i) v += s_all[i][m];
        float* o = of + (int64_t)g * out_gs + tau * d.M + m;
        if (out_gs == 0 && d.G > 1) atomicAdd(o, v);
        else if (accumulate) *o += v; else *o = v;
    }
}

// A4 on a cluster.  Every CTA keeps its slice of (z,y) in registers and its positive entries in shared memory.  The median
// of the positives is found with one fine radix level in the common case: a 4096-bin histogram of bits 30..19 is built
// locally, its non-empty bins are added into ALL eight CTAs' merged histograms through DSMEM, and after one cluster barrier
// every CTA locates the median's bin redundantly.  The few hundred entries of that bin are then broadcast the same way and the
// remaining bits are resolved inside each CTA (block-local radix passes), so no result has to be published: two full
// cluster barriers per call instead of one or two per radix byte.  Degenerate inputs (more than MS_CAND entries in the
// bin, e.g. many equal values) take further 12-bit cluster levels first.
#define MS_BINS 4096
#define MS_CAND 2048
#define MS_THREADS 1024
// rank search in an nb-bin histogram (nb <= 8 * blockDim.x) by the whole block; res[0]=bin, res[1]=count below, res[2]=count in
// bin, res[3]=total; median_rank: rank = lower middle of the total.  Needs hist complete and visible (caller syncs before); ends with a __syncthreads.
__device__ __forceinline__ void block_find_bin(const unsigned int* hist, int nb, unsigned int rank, bool median_rank, unsigned int* wsum, unsigned int* res) {
    const int t = threadIdx.x, lane = t & 31, w = t >> 5, nw = blockDim.x >> 5;
    const int per = (nb + blockDim.x - 1) / blockDim.x;            // <= 8
    unsigned int h[8], sum = 0;
    #pragma unroll
    for (int i = 0; i < 8; ++i) { const int bi = t * per + i; h[i] = (i < per && bi < nb) ? hist[bi] : 0u; sum += h[i]; }
    unsigned int inc = sum;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned int y = __shfl_up_sync(FULLMASK, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    unsigned int base = 0, total = 0;
    for (int i = 0; i < nw; ++i) { const unsigned int x = wsum[i]; if (i < w) base += x; total += x; }
    const unsigned int exc = base + inc - sum;
    if (median_rank) rank = total == 0 ? 0xffffffffu : ((total & 1u) ? total / 2 : total / 2 - 1);   // lower middle entry
    if (rank >= exc && rank < exc + sum) {
        unsigned int c0 = exc; int bi = 0;
        #pragma unroll
        for (; bi < 7; ++bi) { if (c0 + h[bi] > rank) break; c0 += h[bi]; }
        res[0] = (unsigned int)(t * per + bi); res[1] = c0; res[2] = h[bi];
    }
    if (t == 0) res[3] = total;
    __syncthreads();
}

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(MS_THREADS) k_mask_scale_c(const float* __restrict__ z, const float* __restrict__ y,
                                                                                 float* __restrict__ zy, float* __restrict__ med_out, int cap, CscDims d) { PDL_SYNC();
    extern __shared__ float s_dyn[];
    float* s_pos = s_dyn;                                                  // [cap] this CTA's slice: z rows, then y rows
    unsigned int* lhist = reinterpret_cast<unsigned int*>(s_dyn + cap);   // [MS_BINS] local histogram; later scratch
    unsigned int* mhist = lhist + MS_BINS;                                 // [MS_BINS] merged histogram (remote atomics land here)
    float* cand = reinterpret_cast<float*>(mhist + MS_BINS);               // [MS_CAND] merged candidates (remote stores land here)
    __shared__ unsigned int ctl[2];               // [0] candidates reserved so far, [1] min bits of the entries above the bin
    __shared__ unsigned int s_ncand, s_lmin, s_base[CL], wsum[32], res[4];
    cg::cluster_group cluster = cg::this_cluster();
    const int r = (int)cluster.block_rank();
    const int g = blockIdx.x / CL;
    const int lane = threadIdx.x & 31;
    const int rows_total = d.B * d.c;
    const int R = (rows_total + CL - 1) / CL;
    const int row0 = min(rows_total, r * R), row1 = min(rows_total, row0 + R);
    const float* zg = z + ((int64_t)g * rows_total + row0) * d.M;
    const float* yg = y + ((int64_t)g * rows_total + row0) * d.M;
    const int EZ = (row1 - row0) * d.M;
    for (int i = threadIdx.x; i < 2 * MS_BINS; i += blockDim.x) lhist[i] = 0;      // lhist and mhist are adjacent
    if (threadIdx.x == 0) { s_ncand = 0; s_lmin = 0x7f800000u; ctl[0] = 0; ctl[1] = 0x7f800000u; }
    __syncthreads();
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");         // my shared memory is ready for remote adds
    // 1. the slice is read from global memory once into shared memory (z rows then y rows).  Plain loops, not unrolled register
    //    arrays: this kernel runs a few times per step from a cold instruction cache, and with 6280 SASS instructions its run
    //    time was instruction fetch (ncu: 7-9 of 16 warps stalled on no_instruction)
    const int E2 = 2 * EZ;
    #pragma unroll 8
    for (int e = threadIdx.x; e < E2; e += blockDim.x) s_pos[e] = e < EZ ? zg[e] : yg[e - EZ];
    __syncthreads();
    const unsigned int lpos = (unsigned int)E2;
    // 2. cluster radix levels: bits 30..19, 18..7, 6..0
    unsigned int prefix = 0, pmask = 0, krank = 0, npos = 0, cnt = 0;
    int shift = 19, nb = MS_BINS;
    bool first = true, resolved = false;
    for (int lvl = 0; lvl < 3; ++lvl) {
        if (!first) {                                              // rare: clear both histograms, everybody before anybody adds
            for (int i = threadIdx.x; i < 2 * MS_BINS; i += blockDim.x) lhist[i] = 0;
            __syncthreads();
            asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
        }
        for (unsigned e0 = 0; e0 < lpos; e0 += blockDim.x) {
            const unsigned e = e0 + threadIdx.x;
            const float f = e < lpos ? s_pos[e] : 0.f;
            const unsigned int b = __float_as_uint(f);
            if (f > 0.f && (b & pmask) == prefix) atomicAdd(&lhist[(b >> shift) & (unsigned)(nb - 1)], 1u);
        }
        __syncthreads();
        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");       // every CTA's mhist is zeroed
        for (int i = threadIdx.x; i < nb; i += blockDim.x) {
            const unsigned int c = lhist[i];
            if (c) {
                #pragma unroll
                for (int q = 0; q < CL; ++q) atomicAdd(cluster.map_shared_rank(&mhist[i], (r + q) & (CL - 1)), c);
            }
        }
        cluster.sync();                                            // merged histogram complete in every CTA
        block_find_bin(mhist, nb, krank, first, wsum, res);
        if (first) {
            npos = res[3];
            if (npos == 0) break;
            krank = (npos & 1u) ? npos / 2 : npos / 2 - 1;
            first = false;
        }
        const unsigned int bin = res[0];
        krank -= res[1]; cnt = res[2];
        prefix |= bin << shift; pmask |= (unsigned)(nb - 1) << shift;
        __syncthreads();                                           // res is reused
        if (cnt <= MS_CAND) break;
        if (shift == 0) { resolved = true; break; }                // all 31 bits fixed: every entry of the bin is the same value
        if (shift == 19) { shift = 7; nb = MS_BINS; } else { shift = 0; nb = 128; }
    }
    float med = -INFINITY;
    if (npos > 0) {                                                // cluster-uniform
        // 3. broadcast the bin's entries (and the smallest entry above the bin) to every CTA
        unsigned int* lc = lhist;                                  // local candidate list (lhist is no longer needed)
        unsigned int mn = 0x7f800000u;
        for (unsigned e0 = 0; e0 < lpos; e0 += blockDim.x) {
            const unsigned e = e0 + threadIdx.x;
            const float f = e < lpos ? s_pos[e] : 0.f;
            const unsigned int b = __float_as_uint(f);
            const bool in = f > 0.f && (b & pmask) == prefix;
            if (f > 0.f && (b & pmask) > prefix) mn = min(mn, b);
            if (!resolved) {
                const unsigned mk = __ballot_sync(FULLMASK, in);
                unsigned base = 0;
                if (lane == 0 && mk) base = atomicAdd(&s_ncand, __popc(mk));
                base = __shfl_sync(FULLMASK, base, 0);
                if (in) lc[base + __popc(mk & ((1u << lane) - 1u))] = b;
            }
        }
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(FULLMASK, mn, o));
        if (lane == 0 && mn != 0x7f800000u) atomicMin(&s_lmin, mn);
        __syncthreads();
        const unsigned int nc = s_ncand;
        if (threadIdx.x < CL) {
            const int dst = threadIdx.x;
            if (nc) s_base[dst] = atomicAdd(cluster.map_shared_rank(&ctl[0], dst), nc);
            if (s_lmin != 0x7f800000u) atomicMin(cluster.map_shared_rank(&ctl[1], dst), s_lmin);
        }
        __syncthreads();
        for (unsigned i = threadIdx.x; i < nc * CL; i += blockDim.x) {
            const int dst = (int)(i / nc); const unsigned j = i - dst * nc;
            cluster.map_shared_rank(cand, dst)[s_base[dst] + j] = __uint_as_float(lc[j]);
        }
        cluster.sync();                                            // candidates complete in every CTA; nothing remote after this
        // 4. block-local radix passes over the remaining low bits of the candidates
        const unsigned int kin = krank;                            // ascending rank of the median entry inside the bin
        unsigned int v1b = prefix;
        if (!resolved) {
            unsigned int lowfix = 0, lowmask = 0;
            int rem = shift;
            while (rem > 0) {
                const int nbits = rem < 10 ? rem : 10, sh = rem - nbits, nbin = 1 << nbits;
                for (int i = threadIdx.x; i < nbin; i += blockDim.x) lhist[i] = 0;
                __syncthreads();
                for (unsigned e0 = 0; e0 < cnt; e0 += blockDim.x) {
                    const unsigned e = e0 + threadIdx.x;
                    const unsigned int b = e < cnt ? __float_as_uint(cand[e]) : 0u;
                    hist_add(lhist, e < cnt && (b & lowmask) == lowfix, (b >> sh) & (unsigned)(nbin - 1));
                }
                __syncthreads();
                block_find_bin(lhist, nbin, krank, false, wsum, res);
                lowfix |= res[0] << sh; lowmask |= (unsigned)(nbin - 1) << sh; krank -= res[1];
                __syncthreads();
                rem = sh;
            }
            v1b |= lowfix;
        }
        const float v1 = __uint_as_float(v1b);
        if (npos & 1u) med = v1;
        else {
            // second middle value = entry of ascending rank kin+1: a copy of v1, else the next candidate, else the smallest entry above the bin
            unsigned int le = 0, mn2 = 0x7f800000u;
            if (!resolved)
                for (unsigned e = threadIdx.x; e < cnt; e += blockDim.x) { const unsigned int b = __float_as_uint(cand[e]); if (b <= v1b) ++le; else mn2 = min(mn2, b); }
            #pragma unroll
            for (int o = 16; o > 0; o >>= 1) { le += __shfl_xor_sync(FULLMASK, le, o); mn2 = min(mn2, __shfl_xor_sync(FULLMASK, mn2, o)); }
            if (threadIdx.x == 0) { res[0] = 0; res[1] = 0x7f800000u; }
            __syncthreads();
            if (lane == 0) { if (le) atomicAdd(&res[0], le); atomicMin(&res[1], mn2); }
            __syncthreads();
            const unsigned int le_all = resolved ? cnt : res[0];
            const unsigned int v2b = (le_all >= kin + 2) ? v1b : (res[1] != 0x7f800000u ? res[1] : ctl[1]);
            med = v1 * 0.5f + __uint_as_float(v2b) * 0.5f;       // Statistics.middle(a, b) = a/2 + b/2
        }
    }
    if (r == 0 && threadIdx.x == 0) med_out[g] = med;
    // 5. apply the mask to the CTA's slice
    float* og = zy + ((int64_t)g * rows_total + row0) * d.M2;
    #pragma unroll 2
    for (int e = threadIdx.x; e < E2; e += blockDim.x) {
        const int ee = e < EZ ? e : e - EZ;
        const int np = ee / d.M, m = ee - np * d.M;
        const float f = s_pos[e];
        og[(int64_t)np * d.M2 + (e < EZ ? 0 : d.M) + m] = f >= med ? d.mf * f : 0.f;
    }
}
