// Positions -> count matrices on the GPU (SURVEY §8f-4): for every occurrence (motif, sequence, start, strand) the bases
// under the motif are added to that motif's 4 x len count matrix; reverse-strand occurrences add the reverse complement
// (reverse(onehot_code): both dims reversed).  Replaces the host loops of
//   posdicts2countmats / msa_add!   inference/_h6_positions2countmat.jl:7-54
//   obtain_count_matrices           inference/_3_make_pfms.jl:28-46
//   enriched_keys2motifs (counts)   inference/_s1_make_motifs.jl:234-259
// which slice the one-hot Float32 data matrix per occurrence.  Counts are exact integers here; the host converts them
// to the reference's Float32 / Float16 matrices.
#include "common.cuh"

__global__ void __launch_bounds__(256) countmat_kernel(const uint32_t* __restrict__ words, int64_t rowwords, int64_t Lb, int64_t N,
                                                       const mb200_site* __restrict__ sites, int64_t n_sites,
                                                       const int32_t* __restrict__ lens, int32_t maxlen,
                                                       unsigned int* __restrict__ counts, unsigned int* __restrict__ bad) {
    // one thread per (site, column); maxlen columns per site keep the mapping division-free per warp
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t si = t / maxlen;
    const int j = (int)(t - si * maxlen);
    if (si >= n_sites) return;
    const mb200_site s = sites[si];
    const int len = lens[s.motif];
    if (j >= len) return;
    if (s.seq >= N || (int64_t)s.pos + len > Lb) { if (j == 0) atomicAdd(bad, 1u); return; }
    const int64_t p = (int64_t)s.pos + j;
    const uint32_t b = (words[(int64_t)s.seq * rowwords + (p >> 4)] >> ((p & 15) * 2)) & 3u;
    const int col = s.comp ? len - 1 - j : j;
    const uint32_t base = s.comp ? 3u - b : b;
    atomicAdd(&counts[((int64_t)s.motif * maxlen + col) * 4 + base], 1u);
}

extern "C" int32_t mb200_count_matrices(mb200_ctx* ctx, const mb200_seqs* seqs, const mb200_site* sites, int64_t n_sites,
                                        const int64_t* lens, int32_t K, int32_t maxlen, uint32_t* counts) {
    if (!ctx) return MB200_E_INVALID;
    if (!seqs || !lens || !counts || K <= 0 || maxlen <= 0 || n_sites < 0 || (n_sites > 0 && !sites)) MB_FAIL(ctx, MB200_E_INVALID, "count_matrices: bad arguments");
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    if (seqs->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(seqs)); if (rc) return rc; }
    mb_reset_timing(ctx);
    std::vector<int32_t> h_lens(K);
    for (int k = 0; k < K; ++k) {
        if (lens[k] < 1 || lens[k] > maxlen) MB_FAIL(ctx, MB200_E_INVALID, "count_matrices: motif %d has length %lld outside [1, %d]", k, (long long)lens[k], maxlen);
        h_lens[k] = (int32_t)lens[k];
    }
    for (int64_t i = 0; i < n_sites; ++i)
        if (sites[i].motif >= (uint32_t)K) MB_FAIL(ctx, MB200_E_INVALID, "count_matrices: site %lld names motif %u (K=%d)", (long long)i, sites[i].motif, K);
    if (seqs->ragged) {                  // the kernel checks against Lb; a row of a ragged store ends at its own length
        int64_t bad = 0;
        for (int64_t i = 0; i < n_sites; ++i)
            bad += sites[i].seq < (uint64_t)seqs->N && (int64_t)sites[i].pos + lens[sites[i].motif] > seqs->hlens[sites[i].seq];
        if (bad) MB_FAIL(ctx, MB200_E_INVALID, "count_matrices: %lld sites fall outside their sequence", (long long)bad);
    }
    const size_t cbytes = (size_t)K * maxlen * 4 * 4;
    const size_t off_cnt = 0, off_bad = (cbytes + 255) & ~(size_t)255, off_lens = off_bad + 256;
    const size_t off_sites = off_lens + (((size_t)K * 4 + 255) & ~(size_t)255);
    int rc = mb_ensure_buf(ctx, 6, off_sites + (size_t)std::max<int64_t>(n_sites, 1) * sizeof(mb200_site)); if (rc) return rc;
    uint8_t* base = (uint8_t*)ctx->bufs[6];
    MbTimers tm(ctx);
    const int tt = tm.begin(T_TOTAL);
    MB_CUDA(ctx, cudaMemsetAsync(base, 0, off_lens, ctx->stream));
    const int th = tm.begin(T_H2D);
    MB_CUDA(ctx, cudaMemcpyAsync(base + off_lens, h_lens.data(), (size_t)K * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (n_sites) MB_CUDA(ctx, cudaMemcpyAsync(base + off_sites, sites, (size_t)n_sites * sizeof(mb200_site), cudaMemcpyHostToDevice, ctx->stream));
    tm.end(th);
    if (n_sites) {
        const int64_t threads = n_sites * maxlen;
        const int tk = tm.begin(T_COUNT);
        countmat_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(seqs->words, seqs->rowwords, seqs->Lb, seqs->N,
                                                                                 (const mb200_site*)(base + off_sites), n_sites,
                                                                                 (const int32_t*)(base + off_lens), maxlen,
                                                                                 (unsigned int*)(base + off_cnt), (unsigned int*)(base + off_bad));
        tm.end(tk);
        ctx->launches[T_COUNT] += 1;
        MB_CUDA(ctx, cudaGetLastError());
    }
    unsigned int h_bad = 0;
    const int td = tm.begin(T_D2H);
    MB_CUDA(ctx, cudaMemcpyAsync(counts, base + off_cnt, cbytes, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaMemcpyAsync(&h_bad, base + off_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    tm.end(td); tm.end(tt);
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    tm.collect();
    if (h_bad) MB_FAIL(ctx, MB200_E_INVALID, "count_matrices: %u sites fall outside their sequence", h_bad);
    return MB200_OK;
}
