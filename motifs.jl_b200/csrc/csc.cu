// Unrolled convolutional-sparse-coding network: forward, hand-derived reverse pass, AdaBelief, code retrieval.
//
// Reference being replaced (paths under the reference's src/):
//   model.jl:330-395  ADMM_XYZ / ADMM_DF / forward_pass_return_loss   (forward)
//   train.jl:42-46    gradient(ps) do ... end ; Flux.Optimise.update!  (reverse pass + AdaBelief)
//   train.jl:47-52    l1 early-stop statistic
//   inference/_1_code_retrieval.jl:33-56  code_retrieval
//
// The forward pass is recorded once as a tape of ~100 primitive ops over statically allocated buffers; the reverse
// pass replays the tape backwards with each op's adjoint (csc_kernels.cuh).  Shapes are static, selections
// (batch median, per-sequence top-q) are computed on the device, so a whole step is a fixed kernel sequence with
// no host synchronisation inside — it is captured into a CUDA graph and replayed per step.
#include "common.cuh"
#include "csc_kernels.cuh"
#include "tc_corr2d.cuh"
#include "csc_batched.cuh"
#include "csc_fused.cuh"
#include <algorithm>
#include <cstring>
#include <cstdlib>
#include <functional>
#include <map>

#define IDX_RING 8

namespace {

struct Buf { size_t off = 0; size_t n = 0; };            // offsets in floats into the data / grad arenas

struct Op {
    std::function<void(cudaStream_t)> fwd, bwd;
    const char* name;
    int branch = 0;      // 1: runs on the aux stream (a parallel branch between a fork and a join marker)
    int kind = 0;        // 0 kernel op, 1 fork marker, 2 join marker
};

}  // namespace

struct mb200_csc {
    mb200_ctx* ctx = nullptr;
    CscDims d{};
    mb200_hparams hp{};
    int64_t n_train = 0, n_total = 0, n_scalar_train = 0;
    // parameter storage (raw, Flux.params order + 3 warm-up scalars), gradients, AdaBelief state
    float *p_raw = nullptr, *g_raw = nullptr, *mt = nullptr, *st = nullptr;
    int64_t step_count = 0;
    // arenas
    float *data = nullptr, *grad = nullptr;
    size_t arena = 0;
    uint8_t* bits = nullptr; size_t bits_n = 0;          // top-q bitmasks
    int n_lists = 0;                                     // ordered non-zero lists of the x-role tensors (x and d g)
    int32_t* lcnt = nullptr; uint16_t* lidx = nullptr; float* lval = nullptr;
    int mask_cap = 0; int ms_cluster_maxg = 32;             // groups from which the batch median runs as one CTA per group instead of one cluster per group
    cudaStream_t aux = nullptr;                          // second capture stream: independent adjoint kernels / D-F branches run in parallel
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_fork2 = nullptr, ev_join2 = nullptr;
    bool in_branch = false;                              // set while replaying ops of a forked branch (no nested forking)
    uint8_t* bases = nullptr;
    int64_t* idx_dev = nullptr;
    int64_t* idx_pinned = nullptr;                       // ring of IDX_RING slots of NS indices (a step may still be copying the previous one)
    int ring = 0;
    int64_t* idx_identity_dev = nullptr;                 // 0..NS-1, for batches that arrive from the host
    uint32_t* batch_words = nullptr;                     // NS packed sequences of a host-supplied batch
    uint32_t* batch_pinned = nullptr;
    float* host_out = nullptr;                           // pinned: loss[G*3], l1
    std::vector<Op> tape;
    std::map<std::string, Buf> named;
    // raw-vector offsets
    int64_t off_lam, off_kaps, off_eta, off_om, off_kap, off_D, off_F, off_rho, off_mu, off_warm;
    ScalarSegs segs;
    int64_t graph_kernels = 0;
    // effective-scalar slots (index into sc buffer)
    Buf sc; Buf Deff, Feff, Fnrm0, loss;
    int i_lam0, i_kaps0, i_eta0, i_om0, i_kap0, i_rho0, i_mu0, i_lam_w, i_eta_w, i_om_w;
    bool xyz_only = false;
    bool tensor = false;                                 // forward-only handle using the tcgen05 BF16 path for corr2d
    __nv_bfloat16 *tc_A = nullptr, *tc_F = nullptr; int tc_tiles = 0, tc_ld = 104;
    size_t tc_smem3 = 0; int64_t tc_arows = 0;
    C2sCfg c2s; bool no_c2s = false;                         // register-window corr2d (k_corr2d_s) configuration of this shape
    bool batched = false; float* Ft_scratch = nullptr; float* Ft_scratch2 = nullptr; float* Ft_eff = nullptr;      // one-CTA-per-sequence kernels (csc_batched.cuh) for many-group shapes      // tap-grouped kernel (k_corr2d_tc3)
    cudaGraph_t graph = nullptr; cudaGraphExec_t gexec = nullptr; bool graph_ok = false;
    const uint32_t* graph_words = nullptr; int64_t graph_rowwords = 0;
    const uint32_t* last_words = nullptr; int64_t last_rowwords = 0; const int64_t* last_idx = nullptr;      // batch of the last training step (fused_fallback)
    // fused persistent forward kernel (csc_fused.cuh): plan = arena offsets of the tape's buffers, sync area, eligibility
    FzPlan fz{}; bool fused = false, no_fused = false; size_t fz_smem = 0; int fz_nmed = 0;
    uint8_t* fz_sync = nullptr; size_t fz_sync_bytes = 0, fz_zero_bytes = 0; FzBufs fzb{};
    bool fused_bwd = false; size_t fzb_smem = 0; FzBwd fzw{}; float* fz_bwd_buf = nullptr; unsigned int* fz_err_host = nullptr;
    bool fused_bwd_df = false, no_fused_df = false; size_t fzd_smem = 0;      // loss + ADMM_DF reverse pass as one kernel (needs fused_bwd)
    size_t op_xyz_begin = 0, op_xyz_end = 0;                // tape ops of the ADMM_XYZ passes: [begin, end)
    Buf zero_al{}, zero_be{};
    std::vector<SlotRange> slots; SlotRange* slots_dev = nullptr;      // block partials of the scalar adjoints (k_sum_slots)
    size_t grad_extra = 0;          // floats of the grad arena past `arena`: the slices and slots above, which the data arena has no use for
};

namespace {

struct Builder {
    mb200_csc* s;
    size_t cursor = 0;
    size_t bit_cursor = 0;
    int n_lists = 0;
    Buf alloc(size_t n, const char* name = nullptr) {
        Buf b; b.off = cursor; b.n = n; cursor += (n + 63) & ~(size_t)63;
        if (name) s->named[name] = b;
        return b;
    }
};

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

// every kernel of the step is launched through lk().  MB200_PDL=1 adds the programmatic-dependent-launch attribute (each kernel
// begins with griddepcontrol.wait); measured on B200 it does not shorten the captured step (1.27 vs 1.26 ms: the graph's
// node-to-node gaps are already small next to the kernels' own run time), so it is off by default.
static int g_pdl = -1;
static thread_local int64_t g_lk_count = 0;      // kernels enqueued through lk() by this thread
template <typename... KA, typename... A>
inline void lk(void (*k)(KA...), dim3 g, dim3 b, size_t smem, cudaStream_t q, A&&... a) {
    if (g_pdl < 0) { const char* e = getenv("MB200_PDL"); g_pdl = (e && e[0] == '1') ? 1 : 0; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = g; cfg.blockDim = b; cfg.dynamicSmemBytes = smem; cfg.stream = q;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = g_pdl;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, k, static_cast<KA>(a)...);
    ++g_lk_count;
}

}  // namespace

#define D_(b) (s->data + (b).off)
#define G_(b) (s->grad + (b).off)

// Records the whole network.  xyz_only = forward ADMM_XYZ without loss (code retrieval).
static void build_tape(mb200_csc* s, bool xyz_only) {
    const CscDims d = s->d;
    Builder B{s};
    const int64_t nZ = (int64_t)d.NS * d.c * d.M, nZY = (int64_t)d.NS * d.c * d.M2, nX = (int64_t)d.NS * d.l * d.K, nS = (int64_t)d.NS * d.L4;
    const int64_t nD = (int64_t)d.f_len * d.M, nF = (int64_t)d.h * d.M2 * d.K;
    const int n_sc = 3 * d.npx + d.npx + 3 * d.npd + 3;       // lam, eta, om, rho per xyz pass; kaps, kap, mu per df pass; 3 warm
    s->sc = B.alloc(n_sc);
    // scalar slot order = raw order of the scalar arrays, then warm-ups: lam[npx] kaps[npd] eta[npx] om[npx] kap[npd] rho[npx] mu[npd] | lam_w eta_w om_w
    s->i_lam0 = 0; s->i_kaps0 = d.npx; s->i_eta0 = s->i_kaps0 + d.npd; s->i_om0 = s->i_eta0 + d.npx; s->i_kap0 = s->i_om0 + d.npx;
    s->i_rho0 = s->i_kap0 + d.npd; s->i_mu0 = s->i_rho0 + d.npx; s->i_lam_w = s->i_mu0 + d.npd; s->i_eta_w = s->i_lam_w + 1; s->i_om_w = s->i_eta_w + 1;
    {
        const int64_t ro[8] = {s->off_lam, s->off_kaps, s->off_eta, s->off_om, s->off_kap, s->off_rho, s->off_mu, s->off_warm};
        const int ei[8] = {s->i_lam0, s->i_kaps0, s->i_eta0, s->i_om0, s->i_kap0, s->i_rho0, s->i_mu0, s->i_lam_w};
        const int nn[8] = {d.npx, d.npd, d.npx, d.npx, d.npd, d.npx, d.npd, 3};
        for (int i = 0; i < 8; ++i) { s->segs.raw_off[i] = (int)ro[i]; s->segs.eff_idx[i] = ei[i]; s->segs.n[i] = nn[i]; }
        s->segs.nseg = 8;
    }
    s->Deff = B.alloc(nD, "D0"); s->Feff = B.alloc(nF, "F0"); s->Fnrm0 = B.alloc(d.K);
    s->loss = B.alloc((size_t)d.G * 3 + 4 + d.K, "loss");       // per-group {loss, rec, syn}, then the K per-filter terms of l1(F)
    // The reverse pass adds no shared adjoint with float atomics, whose order (and so the rounding) changes from run to run: the adjoints
    // of the prepared D and F get one slice per group, the warm-up's adjoint of D one slice per sequence, the scalar adjoints one slot per
    // block, and the reverse of prep sums them in a fixed order first (k_sum_slices, k_sum_slots).  Only shapes with fl x M > 512 or
    // M > 64 keep the per-element warm-up adjoint k_warm_zy_bwd, which still adds with atomics.
    const bool wz_s = d.fl * d.M <= 512 && d.M <= 64;                 // k_warm_zy_bwd_s: one CTA per sequence
    const int nDs = xyz_only ? 0 : d.G + (wz_s ? d.NS : 0);
    // they live in the grad arena only, past the `arena` floats both arenas share: offsets below are relative to S->grad + S->arena
    s->grad_extra = 0;
    auto galloc = [s](size_t n) -> size_t { const size_t o = s->grad_extra; s->grad_extra += (n + 63) & ~(size_t)63; return o; };
    const size_t gDs = galloc((size_t)nDs * nD), gFs = galloc(xyz_only ? 0 : (size_t)d.G * nF);
    s->slots.clear();
    auto slots = [&](size_t blocks, std::initializer_list<int> idx) -> size_t {      // offset of blocks x |idx| partials
        if (xyz_only) return 0;
        const size_t p = galloc(blocks * idx.size());
        int lane = 0;
        for (int i : idx) s->slots.push_back({i, (int32_t)blocks, (int32_t)idx.size(), 0, (int64_t)(p + lane++)});
        return p;
    };
    mb200_csc* S = s;
#define GX(o) (S->grad + S->arena + (o))
    auto& T = s->tape;
    T.clear();

    // ---- prep (model.jl:153-169) -----------------------------------------------------------------
    {
        const Buf sc = s->sc, De = s->Deff, Fe = s->Feff, Fn0 = s->Fnrm0;
        T.push_back({[=](cudaStream_t q) {
                         // scalar arrays are contiguous in the raw vector except D,F in the middle: copy slot by slot
                         lk(k_prep_scalars, 1, 256, 0, q, S->p_raw, S->data + sc.off, S->segs);
                         lk(k_prep_D, nblk(d.fl * d.M, 128), 128, 0, q, S->p_raw + S->off_D, S->data + De.off, d);
                         lk(k_prep_F, d.K, 256, 0, q, S->p_raw + S->off_F, S->data + Fe.off, S->data + Fn0.off, d);
                         if (S->batched && S->Ft_eff) lk(k_transpose_F, nblk(nF, 256), 256, 0, q, S->data + Fe.off, (int64_t)0, S->Ft_eff, 1, d);     // the prepared filters' transposed copy, read by every k_tconv_b / k_corr2d_kept of the ADMM_XYZ part (forward and reverse)
                         if (S->tensor) lk(k_tc_prep_F3, nblk((int64_t)d.h * TC_CH * d.K * 8, 256), 256, 0, q, S->data + Fe.off, S->tc_F, d.h, d.M2, d.K);
                     },
                     [=](cudaStream_t q) {
                         lk(k_sum_slices, nblk(nD, 256), 256, 0, q, (const float*)GX(gDs), nDs, nD, S->grad + De.off);
                         lk(k_sum_slices, nblk(nF, 256), 256, 0, q, (const float*)GX(gFs), d.G, nF, S->grad + Fe.off);
                         lk(k_sum_slots, n_sc, 256, 0, q, (const float*)GX(0), (const SlotRange*)S->slots_dev, (int)S->slots.size(), S->grad + sc.off);
                         ScalarSegs tr = S->segs; tr.nseg = 7;      // the warm-up scalars (segment 7) are not trained
                         lk(k_prep_scalars_bwd, 1, 256, 0, q, S->p_raw, S->grad + sc.off, S->g_raw, tr);
                         lk(k_prep_D_bwd, nblk(d.fl * d.M, 128), 128, 0, q, S->p_raw + S->off_D, S->data + De.off, S->grad + De.off, S->g_raw + S->off_D, d);
                         lk(k_prep_F_bwd, d.K, 256, 0, q, S->p_raw + S->off_F, S->data + Fe.off, S->data + Fn0.off, S->grad + Fe.off, S->g_raw + S->off_F, d);
                     },
                     "prep"});
    }
    const Buf sc = s->sc, De = s->Deff, Fe = s->Feff;
    float* const SC = nullptr; (void)SC;
    // where the reverse pass adds the adjoint of filter f (group stride gs): the shared prepared D and F go to their per-group slices
    auto gfilt = [=](Buf f, int64_t gs) -> std::pair<float*, int64_t> {
        if (gs == 0 && f.off == De.off) return {GX(gDs), nD};
        if (gs == 0 && f.off == Fe.off) return {GX(gFs), nF};
        return {S->grad + f.off, gs};
    };
#define SCP (S->data + sc.off)

    // helpers that append one op each -------------------------------------------------------------
    const bool fastK = (d.K == 24), fastM = (d.M <= 64);
#define LCNT(L) (S->lcnt + (size_t)(L) * d.NS)
#define LIDX(L) (S->lidx + (size_t)(L) * d.NS * LIST_CAP)
#define LVAL(L) (S->lval + (size_t)(L) * d.NS * LIST_CAP)
    auto run_corr2d = [=](const float* A, const float* filt, int64_t gs, float* out, int acc, cudaStream_t q) {
        if (S->tensor && gs == 0 && !acc) {
            const int64_t rows = (int64_t)d.NS * d.c;
            lk(k_tc_prep_A3, nblk(rows * (TC_CH - 1), 256), 256, 0, q, A, S->tc_A, rows, S->tc_arows, d.M2);
            lk(k_corr2d_tc3<24, 3>, std::min(S->tc_tiles, S->ctx->sm_count), TC3_THREADS, S->tc_smem3, q, S->tc_A, S->tc_arows, S->tc_F, out, rows, S->tc_tiles, d);
            return;
        }
        // one CTA per sequence wins from ~190 sequences up (measured)
        if (S->batched && d.G >= 32 && S->c2s.tr && !S->no_c2s) {
            if (S->c2s.tr == 6) lk(k_corr2d_s<6, 12>, d.NS / S->c2s.spc, S->c2s.threads, S->c2s.smem, q, A, filt, gs, out, acc, S->c2s.spc, S->c2s.js, S->c2s.ldr, d);
            else lk(k_corr2d_s<8, 12>, d.NS / S->c2s.spc, S->c2s.threads, S->c2s.smem, q, A, filt, gs, out, acc, S->c2s.spc, S->c2s.js, S->c2s.ldr, d);
        }
        else if (S->batched && d.G >= 32 && fastK && d.M2 * 24 <= C2B_PRE * 4 * 64) {
            const int ntile = ((d.l + 3) / 4) * 3;            // 4-row x 8-filter register tiles of a sequence
            lk(k_corr2d_b<24>, d.NS, std::min(C2B_THREADS, std::max(64, (ntile + 31) / 32 * 32)), corr2d_b_smem(d, 24), q, A, filt, gs, out, acc, d);
        }
        else if (fastK) lk(k_corr2d_w<24, 4>, d.NS * ((d.l + 3) / 4), 128, 0, q, A, filt, gs, out, acc, d);
        else lk(k_corr2d, nblk(nX, 128), 128, 0, q, A, filt, gs, out, acc, d);
    };
    // D-layer forms: per-output kernels for a single reference batch, one CTA per sequence when the launch holds many groups
    const bool batched = S->batched;
    const size_t smem_rb = recon_b_smem(d), smem_cb = corr_sig_b_smem(d), smem_tb = (size_t)d.c * d.M2 * 4;
    auto run_recon = [=](const float* ca, const float* cb, const float* filt, int64_t gs, float* out, int acc, cudaStream_t q) {
        if (batched) lk(k_recon_b, d.NS, RB_THREADS, smem_rb, q, ca, cb, filt, gs, out, acc, d);
        else lk(k_recon, nblk(nS * 32, 256), 256, 0, q, ca, cb, filt, gs, out, acc, d);
    };
    auto run_corr_sig = [=](const float* sig, float sgn, const float* filt, int64_t gs, float* oa, float* ob, int acc, cudaStream_t q) {
        if (batched) lk(k_corr_sig_b, d.NS, RB_THREADS, smem_cb, q, sig, S->bases, sgn, filt, gs, oa, ob, acc, d);
        else lk(k_corr_sig, nblk(nZ, 256), 256, 0, q, sig, S->bases, sgn, filt, gs, oa, ob, acc, d);
    };
    auto run_dgrad = [=](const float* ca, const float* cb, const float* sig, float sgn, float* of, int64_t ogs, int acc, cudaStream_t q) {
        // many groups: one CTA per group with a 4-lag x 2-filter register tile (the per-lag kernels re-read the codes 32 times)
        if (batched && fastM && d.f_len == 32 && (d.M & 1) == 0 && dgrad_s_smem(d) + 9216 <= S->ctx->smem_optin && !S->no_c2s) lk(k_dgrad_s, dim3(d.G, DGS_SLICES), DG_THREADS, dgrad_s_smem(d), q, ca, cb, sig, S->bases, sgn, of, ogs, acc, d);
        else if (batched && fastM && d.f_len == 32 && (d.M & 1) == 0 && (size_t)d.L4 * 4 <= S->ctx->smem_optin) lk(k_dgrad_g, dim3(d.G, DG_SLICES), DG_THREADS, (size_t)d.L4 * 4, q, ca, cb, sig, S->bases, sgn, of, ogs, acc, d);
        else if (fastM) lk(k_dgrad_c, dim3(d.f_len * CL, d.G), 256, 0, q, ca, cb, sig, S->bases, sgn, of, ogs, acc, d);
        else lk(k_dgrad, dim3(nblk(nD, 128), d.G), 128, 0, q, ca, cb, sig, S->bases, sgn, of, ogs, acc, d);
    };
    auto run_tconv = [=](const float* x, int L, const float* filt, int64_t gs, float* out, int acc, cudaStream_t q) {
        if (batched) {
            const int Gf = gs ? d.G : 1;
            const bool eff = gs == 0 && S->Ft_eff && filt == S->data + Fe.off;       // the transposed copy made right after prep_filters
            if (!eff) lk(k_transpose_F, nblk((int64_t)Gf * nF, 256), 256, 0, q, filt, gs, S->Ft_scratch, Gf, d);
            lk(k_tconv_b, d.NS, RB_THREADS, smem_tb, q, x, LCNT(L), LIDX(L), LVAL(L), (const float*)(eff ? S->Ft_eff : S->Ft_scratch), gs ? nF : (int64_t)0, out, acc, d);
        } else lk(k_tconv_l, d.NS * d.c, 128, 0, q, x, LCNT(L), LIDX(L), LVAL(L), filt, gs, out, acc, d);
    };
    auto run_fgrad = [=](const float* A, const float* x, int L, float* of, int64_t ogs, int acc, cudaStream_t q) {
        // many groups: one CTA per (group, 8 filters); needs 16-byte aligned per-group outputs (ogs, of) when it stores vectors
        if (batched && !S->no_c2s && (d.K & 7) == 0 && (ogs & 3) == 0 && ((uintptr_t)of & 15) == 0)
            lk(k_fgrad_g, dim3(d.G, d.K / 8, (d.h * d.M2 + FG_THREADS - 1) / FG_THREADS), FG_THREADS, 0, q, A, x, LCNT(L), LIDX(L), LVAL(L), of, ogs, acc, d);
        else lk(k_fgrad_l, dim3(d.K, d.h, d.G), 128, 0, q, A, x, LCNT(L), LIDX(L), LVAL(L), of, ogs, acc, d);
    };
    // two independent adjoint kernels of one op: the second runs on the aux stream (a parallel branch of the captured graph)
    auto par2 = [=](cudaStream_t q, const std::function<void(cudaStream_t)>& k1, const std::function<void(cudaStream_t)>& k2) {
        if (S->in_branch || !S->aux) { k1(q); k2(q); return; }
        cudaEventRecord(S->ev_fork, q); cudaStreamWaitEvent(S->aux, S->ev_fork, 0);
        k2(S->aux);
        k1(q);
        cudaEventRecord(S->ev_join, S->aux); cudaStreamWaitEvent(q, S->ev_join, 0);
    };
    std::map<size_t, int> xlist;                 // buffer offset of an x tensor -> list of its data
    std::map<size_t, size_t> xbits;              // buffer offset of an x tensor -> offset of the top-q bitmap that produced it
    // the adjoint of a top-q output is only read on the kept support (k_topq_s_bwd masks it): ~32 dot products per sequence instead of the dense contraction
    auto run_corr2d_kept = [=](const float* A, const float* filt, int64_t gs, size_t bo, float* out, int acc, cudaStream_t q) {
        if (batched && S->Ft_scratch2 && !S->no_c2s) {         // the strided filter reads (4 bytes of every 96) were most of this kernel's time: transpose first
            const int Gf = gs ? d.G : 1;
            const bool eff = gs == 0 && S->Ft_eff && filt == S->data + Fe.off;
            if (!eff) lk(k_transpose_F, nblk((int64_t)Gf * nF, 256), 256, 0, q, filt, gs, S->Ft_scratch2, Gf, d);
            lk(k_corr2d_kept, d.NS, CK_THREADS, (size_t)d.l * d.K * 4, q, A, (const float*)(eff ? S->Ft_eff : S->Ft_scratch2), gs ? nF : (int64_t)0, (const uint8_t*)(S->bits + bo), out, acc, 1, d);
        } else lk(k_corr2d_kept, d.NS, CK_THREADS, (size_t)d.l * d.K * 4, q, A, filt, gs, (const uint8_t*)(S->bits + bo), out, acc, 0, d);
    };
    auto op_recon = [&](Buf ca, Buf cb, Buf filt, int64_t gs, Buf out, const char* nm) {
        T.push_back({[=](cudaStream_t q) { run_recon(S->data + ca.off, S->data + cb.off, S->data + filt.off, gs, S->data + out.off, 0, q); },
                     [=](cudaStream_t q) {
                         // d ca, d cb: corr_sig form with signal = d out ; d filt: dgrad form with signal = d out
                         par2(q, [=](cudaStream_t r) { run_corr_sig(S->grad + out.off, 0.f, S->data + filt.off, gs, S->grad + ca.off, S->grad + cb.off, 1, r); },
                                 [=](cudaStream_t r) { const auto o = gfilt(filt, gs); run_dgrad(S->data + ca.off, S->data + cb.off, S->grad + out.off, 0.f, o.first, o.second, 1, r); });
                     },
                     nm});
    };
    auto op_corr_sig = [&](Buf sig, float sgn, Buf filt, int64_t gs, Buf oa, Buf ob, const char* nm) {
        T.push_back({[=](cudaStream_t q) { run_corr_sig(S->data + sig.off, sgn, S->data + filt.off, gs, S->data + oa.off, S->data + ob.off, 0, q); },
                     [=](cudaStream_t q) {
                         par2(q, [=](cudaStream_t r) { run_recon(S->grad + oa.off, S->grad + ob.off, S->data + filt.off, gs, S->grad + sig.off, 1, r); },
                                 [=](cudaStream_t r) { const auto o = gfilt(filt, gs); run_dgrad(S->grad + oa.off, S->grad + ob.off, S->data + sig.off, sgn, o.first, o.second, 1, r); });
                     },
                     nm});
    };
    auto op_dgrad = [&](Buf ca, Buf cb, Buf sig, float sgn, Buf outG, const char* nm) {      // per-group output
        T.push_back({[=](cudaStream_t q) { run_dgrad(S->data + ca.off, S->data + cb.off, S->data + sig.off, sgn, S->data + outG.off, nD, 0, q); },
                     [=](cudaStream_t q) {
                         // d ca, d cb: corr_sig with filter = dG (per group) ; d sig: recon with filter = dG
                         par2(q, [=](cudaStream_t r) { run_corr_sig(S->data + sig.off, sgn, S->grad + outG.off, nD, S->grad + ca.off, S->grad + cb.off, 1, r); },
                                 [=](cudaStream_t r) { run_recon(S->data + ca.off, S->data + cb.off, S->grad + outG.off, nD, S->grad + sig.off, 1, r); });
                     },
                     nm});
    };
    // out = g feeds exactly one top-q op, whose adjoint writes d g and its non-zero list `glist`
    auto op_corr2d = [&](Buf A, Buf filt, int64_t gs, Buf out, int glist, const char* nm) {
        T.push_back({[=](cudaStream_t q) { run_corr2d(S->data + A.off, S->data + filt.off, gs, S->data + out.off, 0, q); },
                     [=](cudaStream_t q) {
                         par2(q, [=](cudaStream_t r) { run_tconv(S->grad + out.off, glist, S->data + filt.off, gs, S->grad + A.off, 1, r); },
                                 [=](cudaStream_t r) { const auto o = gfilt(filt, gs); run_fgrad(S->data + A.off, S->grad + out.off, glist, o.first, o.second, 1, r); });
                     },
                     nm});
    };
    auto op_tconv = [&](Buf x, Buf filt, int64_t gs, Buf out, const char* nm) {
        const int xl = xlist.at(x.off);
        const size_t xb = xbits.at(x.off);
        T.push_back({[=](cudaStream_t q) { run_tconv(S->data + x.off, xl, S->data + filt.off, gs, S->data + out.off, 0, q); },
                     [=](cudaStream_t q) {
                         par2(q, [=](cudaStream_t r) { run_corr2d_kept(S->grad + out.off, S->data + filt.off, gs, xb, S->grad + x.off, 1, r); },
                                 [=](cudaStream_t r) { const auto o = gfilt(filt, gs); run_fgrad(S->grad + out.off, S->data + x.off, xl, o.first, o.second, 1, r); });
                     },
                     nm});
    };
    auto op_fgrad = [&](Buf A, Buf x, Buf outF, const char* nm) {                               // per-group output
        const int xl = xlist.at(x.off);
        const size_t xb = xbits.at(x.off);
        T.push_back({[=](cudaStream_t q) { run_fgrad(S->data + A.off, S->data + x.off, xl, S->data + outF.off, nF, 0, q); },
                     [=](cudaStream_t q) {
                         par2(q, [=](cudaStream_t r) { run_tconv(S->data + x.off, xl, S->grad + outF.off, nF, S->grad + A.off, 1, r); },
                                 [=](cudaStream_t r) { run_corr2d_kept(S->data + A.off, S->grad + outF.off, nF, xb, S->grad + x.off, 1, r); });
                     },
                     nm});
    };
    const int mask_cap = 2 * ((d.B * d.c + CL - 1) / CL) * d.M;      // floats of dynamic smem per CTA: its slice of rows, z and y
    s->mask_cap = mask_cap;
    auto op_mask_scale = [&](Buf z, Buf y, Buf zy, const char* nm) -> Buf {
        Buf med = B.alloc(d.G);
        // one 8-CTA cluster per group minimises latency (training, few groups); with many groups (batched code retrieval) one CTA per
        // group fills the machine better: 148 groups in flight instead of 18 clusters
        const bool ms_cluster = mask_cap <= MS_MAXV * 512 && d.G < S->ms_cluster_maxg;
        const int ms_cap1 = (int)std::min<int64_t>(2 * (int64_t)d.B * d.c * d.M, 49152);
        T.push_back({[=](cudaStream_t q) {
                         if (ms_cluster) lk(k_mask_scale_c, d.G * CL, MS_THREADS, ((size_t)mask_cap + 2 * MS_BINS + MS_CAND) * 4, q, S->data + z.off, S->data + y.off, S->data + zy.off, S->data + med.off, mask_cap, d);
                         else if (S->batched) lk(k_mask_scale_g, d.G, MG_THREADS, 0, q, S->data + z.off, S->data + y.off, S->data + zy.off, S->data + med.off, d);
                         else lk(k_mask_scale_s, d.G, 1024, (size_t)ms_cap1 * 4, q, S->data + z.off, S->data + y.off, S->data + zy.off, S->data + med.off, ms_cap1, d);
                     },
                     [=](cudaStream_t q) { lk(k_mask_scale_bwd, nblk(nZY, 256), 256, 0, q, S->data + z.off, S->data + y.off, S->data + med.off, S->grad + zy.off, S->grad + z.off, S->grad + y.off, d); },
                     nm});
        return med;
    };
    // returns nothing; registers the data list of xout; `glist` = list id for d g (allocated by the caller)
    size_t last_bo = 0; int last_xl = 0;
    auto op_topq = [&](const Buf* xprev, Buf g, int i_om, float coef, int om_train, Buf xout, int glist, const char* nm) {
        const size_t bo = B.bit_cursor; B.bit_cursor += (size_t)nX;
        const int xl = B.n_lists++;
        last_bo = bo; last_xl = xl;
        xlist[xout.off] = xl; xbits[xout.off] = bo;
        const bool hp_ = xprev != nullptr; const Buf xp = hp_ ? *xprev : Buf{};
        const size_t smem = (size_t)d.l * d.K * 4;
        const size_t om_sl = om_train ? slots((size_t)d.NS, {i_om}) : 0;
        T.push_back({[=](cudaStream_t q) { lk(k_topq_s, d.NS, 256, smem, q, hp_ ? S->data + xp.off : nullptr, S->data + g.off, SCP, i_om, coef, S->data + xout.off, S->bits + bo, LCNT(xl), LIDX(xl), LVAL(xl), d); },
                     [=](cudaStream_t q) { lk(k_topq_s_bwd, d.NS, 256, 0, q, S->bits + bo, S->data + g.off, SCP, i_om, coef, S->grad + xout.off, hp_ ? S->grad + xp.off : nullptr, S->grad + g.off, om_train ? GX(om_sl) : nullptr, om_train, LCNT(glist), LIDX(glist), LVAL(glist), d); },
                     nm});
    };

    // ---- warm-up (model.jl:224-232) --------------------------------------------------------------
    Buf z = B.alloc(nZ), y = B.alloc(nZ);
    T.push_back({[=](cudaStream_t q) { lk(k_warm_zy, nblk(nZ, 256), 256, 0, q, S->bases, S->data + De.off, SCP, S->i_eta_w, S->i_lam_w, S->data + z.off, S->data + y.off, d); },
                 [=](cudaStream_t q) {
                     if (wz_s) lk(k_warm_zy_bwd_s, d.NS, 512, 0, q, S->bases, SCP, S->i_eta_w, S->data + z.off, S->data + y.off, S->grad + z.off, S->grad + y.off, GX(gDs + (size_t)d.G * nD), d);
                     else lk(k_warm_zy_bwd, nblk(nZ, 256), 256, 0, q, S->bases, SCP, S->i_eta_w, S->data + z.off, S->data + y.off, S->grad + z.off, S->grad + y.off, S->grad + De.off, d);
                 },
                 "warm_zy"});
    Buf zy = B.alloc(nZY);
    FzPlan& FP = s->fz;
    memset(&FP, 0, sizeof FP);
    FP.npx = d.npx; FP.npd = d.npd; FP.i_eta_w = s->i_eta_w; FP.i_lam_w = s->i_lam_w; FP.i_om_w = s->i_om_w; FP.forward_only = xyz_only ? 1 : 0;
    FP.sc = (int64_t)sc.off; FP.De = (int64_t)De.off; FP.Fe = (int64_t)Fe.off; FP.z0 = (int64_t)z.off; FP.y0 = (int64_t)y.off; FP.zy0 = (int64_t)zy.off;
    FP.med0 = (int64_t)op_mask_scale(z, y, zy, "warm_mask").off;
    Buf g0 = B.alloc(nX), x = B.alloc(nX);
    { const int gl = B.n_lists++; op_corr2d(zy, Fe, 0, g0, gl, "warm_corr2d"); op_topq(nullptr, g0, s->i_om_w, 1.f, 0, x, gl, "warm_topq"); }
    FP.g0 = (int64_t)g0.off; FP.x0 = (int64_t)x.off; FP.bits0 = (int64_t)last_bo; FP.xl0 = last_xl;
    int cur_xl = last_xl;
    Buf fx = B.alloc(nZY);
    FP.fx0 = (int64_t)fx.off;
    op_tconv(x, Fe, 0, fx, "warm_tconv");
    Buf al{}, be{};
    bool have_dual = false;

    // ---- ADMM_XYZ passes (model.jl:256-268, 347-355) ---------------------------------------------
    s->op_xyz_begin = T.size();
    for (int n = 0; n < d.npx; ++n) {
        const int i_eta = s->i_eta0 + n, i_lam = s->i_lam0 + n, i_rho = s->i_rho0 + n, i_om = s->i_om0 + n;
        Buf rec = B.alloc(nS), gz = B.alloc(nZ), gy = B.alloc(nZ), zn = B.alloc(nZ), yn = B.alloc(nZ);
        op_recon(z, y, De, 0, rec, "recon");
        op_corr_sig(rec, -1.f, De, 0, gz, gy, "corr_sig");
        if (!have_dual) { al = B.alloc(nZ); be = B.alloc(nZ); }      // zero duals (model.jl:338): arenas are zero-filled, never written
        FzPass* XP = n < FZ_MAXPX ? &FP.px[n] : nullptr;
        if (XP) { XP->z_in = (int64_t)z.off; XP->y_in = (int64_t)y.off; XP->fx_in = (int64_t)fx.off; XP->al_in = (int64_t)al.off; XP->be_in = (int64_t)be.off;
                  XP->rec = (int64_t)rec.off; XP->gz = (int64_t)gz.off; XP->gy = (int64_t)gy.off; XP->z_out = (int64_t)zn.off; XP->y_out = (int64_t)yn.off;
                  XP->i_eta = i_eta; XP->i_lam = i_lam; XP->i_rho = i_rho; XP->i_om = i_om; XP->x_in = (int64_t)x.off; XP->xl_in = cur_xl; XP->al_out = -1; XP->be_out = -1; }
        {
            const Buf zc = z, yc = y, fxc = fx, alc = al, bec = be;
            const size_t zy_sl = slots(nblk(nZ, 256), {i_eta, i_lam, i_rho});
            T.push_back({[=](cudaStream_t q) { lk(k_zy_update, nblk(nZ, 256), 256, 0, q, S->data + zc.off, S->data + yc.off, S->data + gz.off, S->data + gy.off, S->data + fxc.off, S->data + alc.off, S->data + bec.off, SCP, i_eta, i_lam, i_rho, S->data + zn.off, S->data + yn.off, d); },
                         [=](cudaStream_t q) { lk(k_zy_update_bwd, nblk(nZ, 256), 256, 0, q, S->data + zc.off, S->data + yc.off, S->data + gz.off, S->data + gy.off, S->data + fxc.off, S->data + alc.off, S->data + bec.off, SCP, i_eta, i_lam, i_rho, S->data + zn.off, S->data + yn.off, S->grad + zn.off, S->grad + yn.off, S->grad + zc.off, S->grad + yc.off, S->grad + gz.off, S->grad + gy.off, S->grad + fxc.off, S->grad + alc.off, S->grad + bec.off, GX(zy_sl), d); },
                         "zy_update"});
        }
        z = zn; y = yn;
        Buf zy2 = B.alloc(nZY), dd = B.alloc(nZY), g = B.alloc(nX), xn = B.alloc(nX), fxn = B.alloc(nZY);
        { const Buf md = op_mask_scale(z, y, zy2, "mask_scale"); if (XP) XP->med = (int64_t)md.off; }
        {
            const Buf fxc = fx, alc = al, bec = be;
            T.push_back({[=](cudaStream_t q) { lk(k_d_build, nblk(nZY, 256), 256, 0, q, S->data + fxc.off, S->data + zy2.off, S->data + alc.off, S->data + bec.off, S->data + dd.off, d); },
                         [=](cudaStream_t q) { lk(k_d_build_bwd, nblk(nZY, 256), 256, 0, q, S->grad + dd.off, S->grad + fxc.off, S->grad + zy2.off, S->grad + alc.off, S->grad + bec.off, d); },
                         "d_build"});
        }
        { const int gl = B.n_lists++; op_corr2d(dd, Fe, 0, g, gl, "corr2d"); op_topq(&x, g, i_om, -1.f, 1, xn, gl, "topq"); }
        s->named["g_last"] = g;
        x = xn;
        if (XP) { XP->dd = (int64_t)dd.off; XP->g = (int64_t)g.off; XP->x_out = (int64_t)xn.off; XP->bits = (int64_t)last_bo; XP->xl_out = last_xl; XP->fx_out = (int64_t)fxn.off; }
        cur_xl = last_xl;
        op_tconv(x, Fe, 0, fxn, "tconv");
        fx = fxn;
        if (n + 1 < d.npx) {      // the duals after the last pass are never read (model.jl:356 returns Z, Y, X)
            Buf an = B.alloc(nZ), bn = B.alloc(nZ);
            const Buf alc = al, bec = be, fxc = fx, zc = z, yc = y;
            T.push_back({[=](cudaStream_t q) { lk(k_dual, nblk(nZ, 256), 256, 0, q, S->data + alc.off, S->data + bec.off, S->data + fxc.off, S->data + zc.off, S->data + yc.off, S->data + an.off, S->data + bn.off, d); },
                         [=](cudaStream_t q) { lk(k_dual_bwd, nblk(nZ, 256), 256, 0, q, S->grad + an.off, S->grad + bn.off, S->grad + alc.off, S->grad + bec.off, S->grad + fxc.off, S->grad + zc.off, S->grad + yc.off, d); },
                         "dual"});
            al = an; be = bn;
            if (XP) { XP->al_out = (int64_t)an.off; XP->be_out = (int64_t)bn.off; }
        }
        have_dual = true;
    }
    s->op_xyz_end = T.size();
    s->named["z"] = z; s->named["y"] = y; s->named["x"] = x;
    if (xyz_only) { s->arena = B.cursor; s->bits_n = B.bit_cursor; s->n_lists = B.n_lists; return; }

    // ---- ADMM_DF (model.jl:362-373) ---------------------------------------------------------------
    Buf zyF = B.alloc(nZY, "zy");
    FP.zyF = (int64_t)zyF.off;
    FP.medF = (int64_t)op_mask_scale(z, y, zyF, "df_mask").off;
    Buf Dc = De, Fc = Fe; int64_t Dgs = 0, Fgs = 0;
    Buf theta{}; bool have_theta = false;
    for (int n = 0; n < d.npd; ++n) {
        const int i_mu = s->i_mu0 + n, i_kap = s->i_kap0 + n, i_kaps = s->i_kaps0 + n;
        // update_D (model.jl:368) and update_F (:369) of one pass touch disjoint tensors: they are recorded as two parallel
        // branches (D chain on the aux stream) between a fork and a join marker, in the forward and in the reverse pass
        T.push_back({nullptr, nullptr, "fork", 0, 1});
        const size_t d_chain_begin = T.size();
        Buf rec = B.alloc(nS), Gm = B.alloc((size_t)d.G * nD), Dn = B.alloc((size_t)d.G * nD);
        FzDf* YP = n < FZ_MAXPD ? &FP.df[n] : nullptr;
        if (YP) { YP->D_in = (int64_t)Dc.off; YP->D_in_gs = (int32_t)Dgs; YP->F_in = (int64_t)Fc.off; YP->F_in_gs = (int32_t)Fgs; YP->rec = (int64_t)rec.off; YP->Gm = (int64_t)Gm.off;
                  YP->Dn = (int64_t)Dn.off; YP->i_mu = i_mu; YP->i_kap = i_kap; YP->i_kaps = i_kaps; }
        op_recon(z, y, Dc, Dgs, rec, "df_recon");
        op_dgrad(z, y, rec, +1.f, Gm, "df_dgrad");                      // R = sumZD + sumYRD + S  ('+S': model.jl:282-285)
        {
            const Buf Dcc = Dc; const int64_t gsc = Dgs;
            const size_t mu_sl = slots(nblk((int64_t)d.G * d.fl * d.M, 128), {i_mu});
            T.push_back({[=](cudaStream_t q) { lk(k_d_update, nblk((int64_t)d.G * d.fl * d.M, 128), 128, 0, q, S->data + Dcc.off, gsc, S->data + Gm.off, SCP, i_mu, S->data + Dn.off, d); },
                         [=](cudaStream_t q) { const auto o = gfilt(Dcc, gsc); lk(k_d_update_bwd, nblk((int64_t)d.G * d.fl * d.M, 128), 128, 0, q, S->data + Dcc.off, gsc, S->data + Gm.off, SCP, i_mu, S->data + Dn.off, S->grad + Dn.off, o.first, o.second, S->grad + Gm.off, GX(mu_sl), d); },
                         "d_update"});
        }
        Dc = Dn; Dgs = nD;
        for (size_t ti = d_chain_begin; ti < T.size(); ++ti) T[ti].branch = 1;
        // update_F
        Buf fxc = B.alloc(nZY), e = B.alloc(nZY), Fg = B.alloc((size_t)d.G * nF), Fn = B.alloc((size_t)d.G * nF), nrm = B.alloc((size_t)d.G * d.K);
        if (YP) { YP->e = (int64_t)e.off; YP->Fg = (int64_t)Fg.off; YP->Fn = (int64_t)Fn.off; YP->nrm = (int64_t)nrm.off; }
        op_tconv(x, Fc, Fgs, fxc, "df_tconv");
        {
            const Buf th = theta; const bool ht = have_theta;
            T.push_back({[=](cudaStream_t q) { lk(k_sub3, nblk(nZY, 256), 256, 0, q, S->data + fxc.off, S->data + zyF.off, ht ? S->data + th.off : nullptr, -1.f, S->data + e.off, nZY); },
                         [=](cudaStream_t q) { lk(k_sub3_bwd, nblk(nZY, 256), 256, 0, q, S->grad + e.off, S->grad + fxc.off, S->grad + zyF.off, ht ? S->grad + th.off : nullptr, -1.f, nZY); },
                         "e_build"});
        }
        op_fgrad(e, x, Fg, "df_fgrad");
        {
            const Buf Fcc = Fc; const int64_t gsc = Fgs;
            const size_t kap_sl = slots((size_t)d.G * d.K, {i_kap, i_kaps});
            T.push_back({[=](cudaStream_t q) { lk(k_f_update, d.G * d.K, 256, 0, q, S->data + Fcc.off, gsc, S->data + Fg.off, SCP, i_kap, i_kaps, S->data + Fn.off, S->data + nrm.off, d); },
                         [=](cudaStream_t q) { const auto o = gfilt(Fcc, gsc); lk(k_f_update_bwd, d.G * d.K, 256, 0, q, S->data + Fn.off, S->data + nrm.off, S->data + Fg.off, SCP, i_kap, i_kaps, S->grad + Fn.off, o.first, o.second, S->grad + Fg.off, GX(kap_sl), d); },
                         "f_update"});
        }
        Fc = Fn; Fgs = nF;
        T.push_back({nullptr, nullptr, "join", 0, 2});
        // theta = theta + FX(X, F_new) - ZY   (only needed by the next pass)
        if (n + 1 < d.npd) {
            Buf fx2 = B.alloc(nZY), thn = B.alloc(nZY);
            op_tconv(x, Fc, Fgs, fx2, "theta_tconv");
            const Buf th = theta; const bool ht = have_theta;
            T.push_back({[=](cudaStream_t q) { lk(k_sub3, nblk(nZY, 256), 256, 0, q, S->data + fx2.off, S->data + zyF.off, ht ? S->data + th.off : nullptr, +1.f, S->data + thn.off, nZY); },
                         [=](cudaStream_t q) { lk(k_sub3_bwd, nblk(nZY, 256), 256, 0, q, S->grad + thn.off, S->grad + fx2.off, S->grad + zyF.off, ht ? S->grad + th.off : nullptr, +1.f, nZY); },
                         "theta"});
            theta = thn; have_theta = true;
            if (YP) { YP->thn = (int64_t)thn.off; YP->has_theta_out = 1; }
        }
    }
    s->named["D"] = Dc; s->named["F"] = Fc;
    // ---- loss (model.jl:310-325) ------------------------------------------------------------------
    Buf recL = B.alloc(nS), fxL = B.alloc(nZY);
    FP.recL = (int64_t)recL.off; FP.fxL = (int64_t)fxL.off; FP.loss = (int64_t)s->loss.off;
    op_recon(z, y, Dc, Dgs, recL, "loss_recon");
    op_tconv(x, Fc, Fgs, fxL, "loss_tconv");
    {
        const Buf ls = s->loss;
        T.push_back({[=](cudaStream_t q) { lk(k_loss, d.G, 1024, 0, q, S->data + recL.off, S->bases, S->data + fxL.off, S->data + zyF.off, S->data + ls.off, d); },
                     [=](cudaStream_t q) { lk(k_loss_bwd, nblk(std::max(nS, nZY), 256), 256, 0, q, S->data + recL.off, S->bases, S->data + fxL.off, S->data + zyF.off, 1.f / (float)d.G, S->grad + recL.off, S->grad + fxL.off, S->grad + zyF.off, d); },
                     "loss"});
    }
    s->arena = B.cursor; s->bits_n = B.bit_cursor; s->n_lists = B.n_lists;
}

#define FZ_BAR_DF 21          // barrier counters: forward kernel [0, 21), DF reverse kernel [21, 42), XYZ reverse kernel [42, 63) (one per group)
#define FZ_BAR_XYZ 42
static int csc_alloc(mb200_ctx* ctx, mb200_csc* s) {
    MB_CUDA(ctx, cudaMalloc(&s->p_raw, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMalloc(&s->g_raw, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMalloc(&s->mt, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMalloc(&s->st, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMemset(s->p_raw, 0, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMemset(s->g_raw, 0, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMemset(s->mt, 0, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMemset(s->st, 0, (size_t)s->n_total * 4));
    MB_CUDA(ctx, cudaMalloc(&s->data, s->arena * 4));
    MB_CUDA(ctx, cudaMemset(s->data, 0, s->arena * 4));
    if (!s->xyz_only) { MB_CUDA(ctx, cudaMalloc(&s->grad, (s->arena + s->grad_extra) * 4)); MB_CUDA(ctx, cudaMemset(s->grad, 0, (s->arena + s->grad_extra) * 4)); }
    if (s->batched) {
        MB_CUDA(ctx, cudaMalloc(&s->Ft_scratch, (size_t)s->d.G * s->d.h * s->d.M2 * s->d.K * 4));
        MB_CUDA(ctx, cudaMalloc(&s->Ft_eff, (size_t)s->d.h * s->d.M2 * s->d.K * 4));
        MB_CUDA(ctx, cudaMalloc(&s->Ft_scratch2, (size_t)s->d.G * s->d.h * s->d.M2 * s->d.K * 4));       // k_corr2d_kept's own copy (it runs beside k_tconv_b on the other branch)
        MB_CUDA(ctx, cudaFuncSetAttribute(k_recon_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)recon_b_smem(s->d)));
        MB_CUDA(ctx, cudaFuncSetAttribute(k_corr_sig_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)corr_sig_b_smem(s->d)));
        MB_CUDA(ctx, cudaFuncSetAttribute(k_tconv_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)s->d.c * s->d.M2 * 4)));
        MB_CUDA(ctx, cudaFuncSetAttribute(k_corr2d_b<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)corr2d_b_smem(s->d, 24)));
        s->c2s = corr2d_s_pick(s->d, ctx->smem_optin);
        s->no_c2s = getenv("MB200_CSC_NO_C2S") != nullptr;      // A/B: keep k_corr2d_b
        if (s->c2s.tr) {
            MB_CUDA(ctx, cudaFuncSetAttribute(k_corr2d_s<6, 12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->c2s.smem));
            MB_CUDA(ctx, cudaFuncSetAttribute(k_corr2d_s<8, 12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->c2s.smem));
        }
    }
    if (!s->slots.empty()) {
        MB_CUDA(ctx, cudaMalloc(&s->slots_dev, s->slots.size() * sizeof(SlotRange)));
        MB_CUDA(ctx, cudaMemcpy(s->slots_dev, s->slots.data(), s->slots.size() * sizeof(SlotRange), cudaMemcpyHostToDevice));
    }
    MB_CUDA(ctx, cudaMalloc(&s->bits, std::max<size_t>(s->bits_n, 16)));
    MB_CUDA(ctx, cudaMalloc(&s->lcnt, (size_t)std::max(1, s->n_lists) * s->d.NS * 4));
    MB_CUDA(ctx, cudaMalloc(&s->lidx, (size_t)std::max(1, s->n_lists) * s->d.NS * LIST_CAP * 2));
    MB_CUDA(ctx, cudaMalloc(&s->lval, (size_t)std::max(1, s->n_lists) * s->d.NS * LIST_CAP * 4));
    MB_CUDA(ctx, cudaMemset(s->lcnt, 0, (size_t)std::max(1, s->n_lists) * s->d.NS * 4));
    if (s->mask_cap <= MS_MAXV * 512) MB_CUDA(ctx, cudaFuncSetAttribute(k_mask_scale_c, cudaFuncAttributeMaxDynamicSharedMemorySize, (s->mask_cap + 2 * MS_BINS + MS_CAND) * 4));
    MB_CUDA(ctx, cudaFuncSetAttribute(k_mask_scale_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::min<int64_t>(2 * (int64_t)s->d.B * s->d.c * s->d.M, 49152) * 4));
    MB_CUDA(ctx, cudaFuncSetAttribute(k_topq_s, cudaFuncAttributeMaxDynamicSharedMemorySize, s->d.l * s->d.K * 4));
    MB_CUDA(ctx, cudaFuncSetAttribute(k_corr2d_kept, cudaFuncAttributeMaxDynamicSharedMemorySize, s->d.l * s->d.K * 4));
    if ((size_t)s->d.L4 * 4 <= ctx->smem_optin) MB_CUDA(ctx, cudaFuncSetAttribute(k_dgrad_g, cudaFuncAttributeMaxDynamicSharedMemorySize, s->d.L4 * 4));
    if (dgrad_s_smem(s->d) + 9216 <= ctx->smem_optin) MB_CUDA(ctx, cudaFuncSetAttribute(k_dgrad_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dgrad_s_smem(s->d)));
    if (s->tensor) {
        const int64_t rows = (int64_t)s->d.NS * s->d.c;
        // the tap-grouped kernel k_corr2d_tc3<K = 24, h/4 = 3> (tc_corr2d.cuh) is the one instantiated shape
        const int R = TC_M + s->d.h - TC_J;
        s->tc_tiles = (int)((rows + TC_VALID - 1) / TC_VALID);
        const size_t arows = (size_t)rows + 2 * TC_M + s->d.h + 8;        // the last tile stays inside the zero padding
        s->tc_arows = (int64_t)arows;
        MB_CUDA(ctx, cudaMalloc(&s->tc_A, arows * s->tc_ld * 2));
        MB_CUDA(ctx, cudaMemset(s->tc_A, 0, arows * s->tc_ld * 2));
        MB_CUDA(ctx, cudaMalloc(&s->tc_F, (size_t)s->d.h * TC_CH * TC_N * 8 * 2));
        s->tc_smem3 = TC3_STAGES * ((((size_t)TC_CH * R * 16) + 1023) & ~(size_t)1023) + (size_t)s->d.h * TC_CH * s->d.K * 16 + 4 * 3 * (TC_J - 1) * (TC_J - 1) * 24 * 4;
        MB_CUDA(ctx, cudaFuncSetAttribute(k_corr2d_tc3<24, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->tc_smem3));
    }
    // ---- fused persistent forward kernel (csc_fused.cuh): the reference's own shapes, all clusters co-resident ----
    {
        const CscDims& d = s->d;
        s->fused = false;
        s->fz_smem = fz::fz_smem_bytes(d.Lb);
        s->fz_nmed = d.npx + 2;
        // a training step with q > LIST_CAP always has code lists the fused reverse pass cannot hold: such handles keep the tape
        const bool shape_ok = d.M == FZ_M && d.K == FZ_K && d.h == FZ_H && d.fl == FZ_FL && d.npx <= FZ_MAXPX && d.npd <= FZ_MAXPD &&
                              d.B * LIST_CAP <= FZ_THREADS && d.B * FZ_CL >= FZ_K && d.c >= FZ_CL && d.l >= 1 && fz::fz_rows(d.c) <= 32 && d.G <= FZ_BAR_DF &&
                              (s->xyz_only || d.q <= LIST_CAP);
        if (!s->no_fused && !s->tensor && shape_ok && s->fz_smem <= ctx->smem_optin) {
            cudaError_t e = cudaFuncSetAttribute(k_csc_fused_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->fz_smem);
#if FZ_CL > 8
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_csc_fused_fwd, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_csc_fused_bwd_xyz, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_csc_fused_bwd_df, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
#endif
            int nclus = 0;
            if (e == cudaSuccess) {
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3((unsigned)(d.NS * FZ_CL)); cfg.blockDim = dim3(FZ_THREADS); cfg.dynamicSmemBytes = s->fz_smem;
                e = cudaOccupancyMaxActiveClusters(&nclus, k_csc_fused_fwd, &cfg);
            }
            if (e != cudaSuccess) { cudaGetLastError(); nclus = 0; }
            s->fused = nclus >= d.NS;                      // every cluster must be resident: the kernel synchronises across them
        }
        if (s->fused) {
            const size_t nmed = (size_t)s->fz_nmed, G = (size_t)d.G;
            const size_t o_bar = 0, o_ctl = 256 + ((G * 4 + 255) & ~(size_t)255), o_hist = o_ctl + ((G * nmed * 16 + 255) & ~(size_t)255);
            const size_t o_cand = o_hist + G * nmed * FZ_NHIST * FZ_BINS * 4;
            const size_t o_part = o_cand + G * nmed * FZ_CAND * 4;
            s->fz_zero_bytes = o_cand;
            s->fz_sync_bytes = o_part + G * (size_t)d.B * FZ_CL * FZ_PART * 4;
            MB_CUDA(ctx, cudaMalloc(&s->fz_sync, s->fz_sync_bytes));
            MB_CUDA(ctx, cudaMemset(s->fz_sync, 0, s->fz_sync_bytes));
            FzBufs& b = s->fzb;
            b.data = s->data; b.bits = s->bits; b.lcnt = s->lcnt; b.lidx = s->lidx; b.lval = s->lval; b.bases = s->bases;
            b.bar = (unsigned int*)(s->fz_sync + o_bar); b.cctl = (unsigned int*)(s->fz_sync + o_ctl); b.hist = (unsigned int*)(s->fz_sync + o_hist);
            b.cand = (float*)(s->fz_sync + o_cand); b.part = (float*)(s->fz_sync + o_part);
            // reverse pass of the XYZ passes as one kernel (training handles only)
            s->fzb_smem = fz::fzb_smem_bytes(d.Lb);
            if (!s->xyz_only && s->fzb_smem <= ctx->smem_optin &&
                cudaFuncSetAttribute(k_csc_fused_bwd_xyz, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->fzb_smem) == cudaSuccess) {
                int nclus = 0;
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3((unsigned)(d.NS * FZ_CL)); cfg.blockDim = dim3(FZ_THREADS); cfg.dynamicSmemBytes = s->fzb_smem;
                if (cudaOccupancyMaxActiveClusters(&nclus, k_csc_fused_bwd_xyz, &cfg) != cudaSuccess) { cudaGetLastError(); nclus = 0; }
                s->fused_bwd = nclus >= d.NS;
            }
            if (s->fused_bwd) {
                const size_t nF = (size_t)d.h * d.M2 * d.K, nD = (size_t)d.f_len * d.M;
                const size_t n_dFp = (size_t)d.NS * nF, n_xch = (size_t)d.NS * FZ_KCAP, n_gsum = 2 * G * (nF + nD + 64);      // second half: group sums of the DF reverse kernel
                MB_CUDA(ctx, cudaMalloc(&s->fz_bwd_buf, (n_dFp + n_xch + n_gsum + 64) * 4));
                MB_CUDA(ctx, cudaMemset(s->fz_bwd_buf, 0, (n_dFp + n_xch + n_gsum + 64) * 4));
                s->fzw.grad = s->grad; s->fzw.dFp = s->fz_bwd_buf; s->fzw.xch = s->fz_bwd_buf + n_dFp; s->fzw.gsum = s->fzw.xch + n_xch;
                s->fzw.err = (unsigned int*)(s->fzw.gsum + n_gsum);
                MB_CUDA(ctx, cudaMallocHost(&s->fz_err_host, 64));
                *s->fz_err_host = 0;
                s->fzd_smem = fz::fzd_smem_bytes(d.Lb);
                if (!s->no_fused_df && s->fzd_smem <= ctx->smem_optin &&
                    cudaFuncSetAttribute(k_csc_fused_bwd_df, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->fzd_smem) == cudaSuccess) {
                    int nclus = 0;
                    cudaLaunchConfig_t cfg = {};
                    cfg.gridDim = dim3((unsigned)(d.NS * FZ_CL)); cfg.blockDim = dim3(FZ_THREADS); cfg.dynamicSmemBytes = s->fzd_smem;
                    if (cudaOccupancyMaxActiveClusters(&nclus, k_csc_fused_bwd_df, &cfg) != cudaSuccess) { cudaGetLastError(); nclus = 0; }
                    s->fused_bwd_df = nclus >= d.NS;
                }
            }
        }
    }
    MB_CUDA(ctx, cudaStreamCreateWithFlags(&s->aux, cudaStreamNonBlocking));
    MB_CUDA(ctx, cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming));
    MB_CUDA(ctx, cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));
    MB_CUDA(ctx, cudaEventCreateWithFlags(&s->ev_fork2, cudaEventDisableTiming));
    MB_CUDA(ctx, cudaEventCreateWithFlags(&s->ev_join2, cudaEventDisableTiming));
    MB_CUDA(ctx, cudaMalloc(&s->bases, (size_t)s->d.NS * s->d.Lb));
    MB_CUDA(ctx, cudaMalloc(&s->idx_dev, (size_t)s->d.NS * 8));
    MB_CUDA(ctx, cudaMallocHost(&s->idx_pinned, (size_t)s->d.NS * 8 * IDX_RING));
    {
        const size_t rw = (size_t)(s->d.Lb + 15) / 16;
        MB_CUDA(ctx, cudaMalloc(&s->idx_identity_dev, (size_t)s->d.NS * 8));
        MB_CUDA(ctx, cudaMalloc(&s->batch_words, ((size_t)s->d.NS * rw + 64) * 4));
        MB_CUDA(ctx, cudaMemset(s->batch_words, 0, ((size_t)s->d.NS * rw + 64) * 4));
        MB_CUDA(ctx, cudaMallocHost(&s->batch_pinned, (size_t)s->d.NS * rw * 4 * IDX_RING));
        std::vector<int64_t> id(s->d.NS);
        for (int i = 0; i < s->d.NS; ++i) id[i] = i;
        MB_CUDA(ctx, cudaMemcpy(s->idx_identity_dev, id.data(), (size_t)s->d.NS * 8, cudaMemcpyHostToDevice));
    }
    MB_CUDA(ctx, cudaMallocHost(&s->host_out, ((size_t)s->d.G * 3 + 8 + s->d.K) * 4));
    return MB200_OK;
}

extern "C" int32_t mb200_csc_create(mb200_ctx* ctx, const mb200_hparams* hp, int64_t Lb, int32_t n_groups, int32_t forward_only, mb200_csc** out) {
    if (!ctx || !hp || !out) return MB200_E_INVALID;
    *out = nullptr;
    if (hp->filter_len < 1 || hp->M < 1 || hp->h < 1 || hp->K < 1 || hp->q < 1 || hp->batch_size < 1 || hp->num_pass_xyz < 1 || hp->num_pass_df < 1 || n_groups < 1)
        MB_FAIL(ctx, MB200_E_INVALID, "csc: bad hyper-parameters");
    const int64_t c = Lb - hp->filter_len + 1, l = c - hp->h + 1;
    if ((int64_t)l * hp->K * 4 > 200 * 1024 || (int64_t)l * hp->K > 65535) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "csc: sequence length %lld too long for the shared-memory top-q", (long long)Lb);
    if (l < 1 || (int64_t)l * hp->K < hp->q) MB_FAIL(ctx, MB200_E_INVALID, "csc: sequence length %lld too short for filter_len %d, h %d, q %d", (long long)Lb, hp->filter_len, hp->h, hp->q);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    mb200_csc* s = new mb200_csc();
    s->no_fused = (forward_only & 0x100) != 0;            // MB200_CSC_NO_FUSED: keep the kernel-per-op tape (A/B tests of the fused step)
    s->no_fused_df = (forward_only & 0x200) != 0;         // MB200_CSC_NO_FUSED_DF: loss / ADMM_DF reverse pass on the tape (A/B tests)
    forward_only &= 0xff;
    s->ctx = ctx; s->hp = *hp; s->xyz_only = forward_only != 0;
    s->tensor = forward_only == 2;
    if (s->tensor && (hp->K != 24 || hp->h != 3 * TC_J || 2 * hp->M > (TC_CH - 1) * 8)) { delete s; MB_FAIL(ctx, MB200_E_UNSUPPORTED, "csc: the tensor-core path is built for K = 24, h = %d and 2M <= %d", 3 * TC_J, (TC_CH - 1) * 8); }
    CscDims& d = s->d;
    d.B = hp->batch_size; d.G = n_groups; d.NS = d.B * d.G; d.Lb = (int)Lb; d.L4 = 4 * (int)Lb; d.c = (int)c; d.l = (int)l;
    d.M = hp->M; d.M2 = 2 * hp->M; d.K = hp->K; d.h = hp->h; d.q = hp->q; d.fl = hp->filter_len; d.f_len = 4 * hp->filter_len;
    d.npx = hp->num_pass_xyz; d.npd = hp->num_pass_df; d.mf = hp->magnifying_factor;
    // raw vector layout = Flux.params(cdl) order (model.jl:67-137): lam[npx] kaps[npd] eta[npx] om[npx] kap[npd] D F rho[npx] mu[npd] | 3 warm-ups
    int64_t o = 0;
    s->off_lam = o; o += d.npx; s->off_kaps = o; o += d.npd; s->off_eta = o; o += d.npx; s->off_om = o; o += d.npx; s->off_kap = o; o += d.npd;
    s->off_D = o; o += (int64_t)d.f_len * d.M; s->off_F = o; o += (int64_t)d.h * d.M2 * d.K; s->off_rho = o; o += d.npx; s->off_mu = o; o += d.npd;
    s->n_train = o; s->off_warm = o; o += 3; s->n_total = o;
    {   // one CTA per sequence pays off once the launch holds enough sequences to fill the machine (MB200_BATCHED_MIN_G overrides)
        const char* e = getenv("MB200_BATCHED_MIN_G");
        const int min_g = e ? atoi(e) : 8;       // measured break-even on B200 (Lb = 100): 8 groups = 48 CTAs
        s->batched = d.G >= min_g && d.f_len == 32 && recon_b_fits(d) && recon_b_smem(d) <= 200 * 1024 && (size_t)d.c * d.M2 * 4 <= 200 * 1024;
    }
    { const char* e = getenv("MB200_MS_CLUSTER_MAXG"); if (e) s->ms_cluster_maxg = atoi(e); }
    build_tape(s, s->xyz_only);
    int rc = csc_alloc(ctx, s);
    if (rc) { delete s; return rc; }
    *out = s;
    return MB200_OK;
}

extern "C" int32_t mb200_csc_destroy(mb200_ctx* ctx, mb200_csc* s) {
    if (!s) return MB200_E_INVALID;
    if (ctx) cudaSetDevice(ctx->device);
    if (s->gexec) cudaGraphExecDestroy(s->gexec);
    if (s->graph) cudaGraphDestroy(s->graph);
    if (s->aux) cudaStreamDestroy(s->aux);
    if (s->ev_fork) { cudaEventDestroy(s->ev_fork); cudaEventDestroy(s->ev_join); cudaEventDestroy(s->ev_fork2); cudaEventDestroy(s->ev_join2); }
    cudaFree(s->p_raw); cudaFree(s->g_raw); cudaFree(s->mt); cudaFree(s->st); cudaFree(s->data); cudaFree(s->grad); cudaFree(s->bits); cudaFree(s->lcnt); cudaFree(s->lidx); cudaFree(s->lval); cudaFree(s->tc_A); cudaFree(s->tc_F); cudaFree(s->Ft_scratch); cudaFree(s->Ft_scratch2); cudaFree(s->Ft_eff); cudaFree(s->fz_sync); cudaFree(s->fz_bwd_buf); cudaFree(s->slots_dev); if (s->fz_err_host) cudaFreeHost(s->fz_err_host);
    cudaFree(s->bases); cudaFree(s->idx_dev); cudaFreeHost(s->idx_pinned); cudaFree(s->idx_identity_dev); cudaFree(s->batch_words); cudaFreeHost(s->batch_pinned); cudaFreeHost(s->host_out);
    delete s;
    return MB200_OK;
}

extern "C" int32_t mb200_csc_n_params(const mb200_csc* s, int64_t* n_trainable, int64_t* n_total) {
    if (!s) return MB200_E_INVALID;
    if (n_trainable) *n_trainable = s->n_train;
    if (n_total) *n_total = s->n_total;
    return MB200_OK;
}

extern "C" int32_t mb200_csc_set_params(mb200_ctx* ctx, mb200_csc* s, const float* p, int64_t n) {
    if (!ctx || !s || !p) return MB200_E_INVALID;
    if (n != s->n_total) MB_FAIL(ctx, MB200_E_INVALID, "csc: expected %lld parameters (trainable %lld + 3 warm-up scalars)", (long long)s->n_total, (long long)s->n_train);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    MB_CUDA(ctx, cudaMemcpyAsync(s->p_raw, p, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
}

extern "C" int32_t mb200_csc_get_params(mb200_ctx* ctx, mb200_csc* s, float* p, int64_t n) {
    if (!ctx || !s || !p) return MB200_E_INVALID;
    if (n != s->n_total) MB_FAIL(ctx, MB200_E_INVALID, "csc: expected %lld parameters", (long long)s->n_total);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    MB_CUDA(ctx, cudaMemcpyAsync(p, s->p_raw, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
}

// the gradient vector as it currently sits on the device: local gradients after mb200_csc_step_begin, the rank-averaged ones after
// mb200_csc_adabelief_step of a ctx with a communicator (tests and bench.py check "all-reduced == mean of the per-rank gradients")
extern "C" int32_t mb200_csc_get_grads(mb200_ctx* ctx, mb200_csc* s, float* g, int64_t n) {
    if (!ctx || !s || !g) return MB200_E_INVALID;
    if (n != s->n_train) MB_FAIL(ctx, MB200_E_INVALID, "csc: expected %lld gradients", (long long)s->n_train);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    MB_CUDA(ctx, cudaMemcpyAsync(g, s->g_raw, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
}

extern "C" int32_t mb200_csc_reset_optimizer(mb200_ctx* ctx, mb200_csc* s) {
    if (!ctx || !s) return MB200_E_INVALID;
    MB_CUDA(ctx, cudaMemsetAsync(s->mt, 0, (size_t)s->n_total * 4, ctx->stream));
    MB_CUDA(ctx, cudaMemsetAsync(s->st, 0, (size_t)s->n_total * 4, ctx->stream));
    s->step_count = 0;
    return MB200_OK;
}

// rank `root`'s parameters, AdaBelief moments and step counter become everybody's (start of data-parallel training: replicas
// that were initialised from different random streams would otherwise apply the averaged gradients to different weights)
extern "C" int32_t mb200_csc_broadcast_params(mb200_ctx* ctx, mb200_csc* s, int32_t root) {
    if (!ctx || !s) return MB200_E_INVALID;
    if (!ctx->comm || ctx->world == 1) return MB200_OK;
    if (root < 0 || root >= ctx->world) MB_FAIL(ctx, MB200_E_INVALID, "csc_broadcast_params: root %d of %d", root, ctx->world);
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = mb_comm_broadcast_bytes(ctx, s->p_raw, (size_t)s->n_total * 4, root); if (rc) return rc;
    rc = mb_comm_broadcast_bytes(ctx, s->mt, (size_t)s->n_total * 4, root); if (rc) return rc;
    rc = mb_comm_broadcast_bytes(ctx, s->st, (size_t)s->n_total * 4, root); if (rc) return rc;
    int64_t sc = s->step_count;
    rc = mb200_comm_broadcast(ctx, &sc, 8, root); if (rc) return rc;      // blocking: also drains the three broadcasts above
    s->step_count = sc;
    return MB200_OK;
}

extern "C" int32_t mb200_csc_device_ptrs(const mb200_csc* s, void** params_dev, void** grads_dev) {
    if (!s) return MB200_E_INVALID;
    if (params_dev) *params_dev = s->p_raw;
    if (grads_dev) *grads_dev = s->g_raw;
    return MB200_OK;
}

// enqueue: gather the batch, forward tape, (optionally) reverse tape.  No host sync inside.
static void run_op(mb200_csc* s, Op& op, bool fwd, cudaStream_t q) {
    auto fork = [&]() { cudaEventRecord(s->ev_fork2, q); cudaStreamWaitEvent(s->aux, s->ev_fork2, 0); s->in_branch = true; };
    auto join = [&]() { cudaEventRecord(s->ev_join2, s->aux); cudaStreamWaitEvent(q, s->ev_join2, 0); s->in_branch = false; };
    if (op.kind == 1) { if (fwd) fork(); else join(); return; }      // in the reverse pass the markers swap roles
    if (op.kind == 2) { if (fwd) join(); else fork(); return; }
    cudaStream_t qq = op.branch ? s->aux : q;
    if (fwd) op.fwd(qq); else op.bwd(qq);
}

// Invariant of the fused kernels' sync area (barrier counters of the three kernels, median histograms and controls): it is all-zero
// whenever a step begins.  The fully fused training step restores that in its last kernel (k_csc_fused_tail); every other fused path
// clears it with memset nodes after the last kernel that used it.  Likewise the adjoint arena: the fully fused step reads only the d x
// slots from it before writing, and those are cleared by their reader (k_csc_fused_bwd_xyz), so it needs no memset per step.
static void launch_fused(mb200_csc* s, int which, cudaStream_t q) {
    const CscDims d = s->d;
    FzBufs fb = s->fzb;
    fb.bases = s->bases; fb.data = s->data; fb.bits = s->bits; fb.lcnt = s->lcnt; fb.lidx = s->lidx; fb.lval = s->lval;
    s->fzw.grad = s->grad;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(d.NS * FZ_CL)); cfg.blockDim = dim3(FZ_THREADS); cfg.stream = q;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (which == 0) { cfg.dynamicSmemBytes = s->fz_smem; cudaLaunchKernelEx(&cfg, k_csc_fused_fwd, s->fz, fb, d); }
    else if (which == 1) {
        fb.bar += FZ_BAR_DF; cfg.dynamicSmemBytes = s->fzd_smem;
        float* gsum2 = s->fzw.gsum + (size_t)d.G * ((size_t)d.h * d.M2 * d.K + (size_t)d.f_len * d.M + 64);
        cudaLaunchKernelEx(&cfg, k_csc_fused_bwd_df, s->fz, fb, s->fzw, gsum2, d);
    } else { fb.bar += FZ_BAR_XYZ; cfg.dynamicSmemBytes = s->fzb_smem; cudaLaunchKernelEx(&cfg, k_csc_fused_bwd_xyz, s->fz, fb, s->fzw, d); }
    ++g_lk_count;
}

// tape = true runs the kernel-per-op tape on a handle built for the fused kernels (fused_fallback)
static void enqueue_step(mb200_csc* s, const uint32_t* words, int64_t rowwords, const int64_t* idx_dev, bool backward, cudaStream_t q, bool tape = false) {
    const CscDims d = s->d;
    const bool fused = s->fused && !tape, fused_bwd = fused && s->fused_bwd, fused_bwd_df = fused_bwd && s->fused_bwd_df;
    const bool fused_all = backward && fused_bwd_df;
    if (fused) {
        // prep_params + unpacking of the batch in one kernel, then the whole forward pass as ONE persistent cooperative kernel
        lk(k_csc_fused_head, d.K + 2 + (unsigned)std::min<int64_t>(8, ((int64_t)d.NS * d.Lb + 255) / 256), 256, 0, q, (const float*)s->p_raw, s->off_D, s->off_F,
           s->data + s->Feff.off, s->data + s->Fnrm0.off, s->data + s->Deff.off, s->data + s->sc.off, s->segs, words, rowwords, idx_dev, s->bases, d);
        launch_fused(s, 0, q);
        if (!fused_all) cudaMemsetAsync(s->fz_sync, 0, s->fz_zero_bytes, q);
    } else {
        lk(k_unpack_bases, nblk((int64_t)d.NS * d.Lb, 256), 256, 0, q, words, rowwords, idx_dev, s->bases, d);
        for (auto& op : s->tape) run_op(s, op, true, q);
    }
    if (backward) {
        if (!fused_all) {
            cudaMemsetAsync(s->grad, 0, (s->arena + s->grad_extra) * 4, q);
            cudaMemsetAsync(s->g_raw, 0, (size_t)s->n_total * 4, q);
        }
        for (size_t i = s->tape.size(); i-- > 0;) {
            if (fused_bwd_df && i >= s->op_xyz_end) {
                // loss, ADMM_DF passes and the final mask in reverse as ONE persistent kernel: leaves d z, d y, d x (kept support) of the
                // final codes for the XYZ kernel below and its share of dD, dF, d scalars in the second half of gsum
                if (i + 1 == s->tape.size()) launch_fused(s, 1, q);
                continue;
            }
            if (fused_bwd && i >= s->op_xyz_begin && i < s->op_xyz_end) {
                if (i + 1 == s->op_xyz_end) {
                    // the reverse pass of all ADMM_XYZ passes and of the warm-up as ONE persistent kernel: reads the adjoints left for the final
                    // z, y, x and adds its share of dD, dF, d scalars to gsum
                    launch_fused(s, 2, q);
                    if (!fused_bwd_df) {            // A/B mode with the DF reverse pass on the tape: add the group sums to the tape's adjoints
                        const int nF = d.h * d.M2 * d.K, nD = d.f_len * d.M, nsc = 3 * d.npx + d.npx + 3 * d.npd + 3;
                        lk(k_csc_fused_finish, nblk(nF + nD + 64, 256), 256, 0, q, (const float*)s->fzw.gsum, d.G, nF, nD, nsc,
                           s->grad + s->Feff.off, s->grad + s->Deff.off, s->grad + s->sc.off);
                    }
                    if (!fused_all) cudaMemsetAsync(s->fz_sync, 0, 256, q);
                }
                continue;
            }
            if (fused_bwd && i >= 1 && i < s->op_xyz_begin) continue;      // the reverse pass of the warm-up is the tail of k_csc_fused_bwd_xyz
            if (fused_all && i == 0) {
                // group sums of both reverse kernels -> adjoint of prep_params -> raw gradient vector; also clears the sync area
                ScalarSegs tr = s->segs; tr.nseg = 7;      // the warm-up scalars (segment 7) are not trained
                const int64_t z16 = (int64_t)(s->fz_zero_bytes / 16);
                lk(k_csc_fused_tail, d.K + 2 + 16, 256, 0, q, (const float*)s->fzw.gsum, 2 * d.G, (const float*)s->p_raw, s->off_D, s->off_F,
                   (const float*)(s->data + s->Feff.off), (const float*)(s->data + s->Fnrm0.off), (const float*)(s->data + s->Deff.off),
                   s->g_raw, tr, reinterpret_cast<uint4*>(s->fz_sync), z16, d);
                continue;
            }
            run_op(s, s->tape[i], false, q);
        }
    }
}

// launches one step on `words` (resident sequence store, or the handle's own buffer holding a host-supplied batch)
static int launch_step(mb200_ctx* ctx, mb200_csc* s, const uint32_t* words, int64_t rowwords, const int64_t* idx_dev, bool backward) {
    if (backward) {                        // the training step is replayed thousands of times: capture it once per source
        s->last_words = words; s->last_rowwords = rowwords; s->last_idx = idx_dev;
        if (!s->graph_ok || s->graph_words != words || s->graph_rowwords != rowwords) {
            if (s->gexec) { cudaGraphExecDestroy(s->gexec); s->gexec = nullptr; }
            if (s->graph) { cudaGraphDestroy(s->graph); s->graph = nullptr; }
            MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            MB_CUDA(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
            const int64_t c0 = g_lk_count;
            enqueue_step(s, words, rowwords, idx_dev, true, ctx->stream);
            s->graph_kernels = g_lk_count - c0;                  // kernel nodes of the captured step
            MB_CUDA(ctx, cudaStreamEndCapture(ctx->stream, &s->graph));
            MB_CUDA(ctx, cudaGraphInstantiate(&s->gexec, s->graph, 0));
            s->graph_ok = true; s->graph_words = words; s->graph_rowwords = rowwords;
        }
        MB_CUDA(ctx, cudaGraphLaunch(s->gexec, ctx->stream));
        ctx->launches[T_CSC] += s->graph_kernels;
    } else {
        const int64_t c0 = g_lk_count;
        enqueue_step(s, words, rowwords, idx_dev, false, ctx->stream);
        ctx->launches[T_CSC] += g_lk_count - c0;
    }
    MB_CUDA(ctx, cudaGetLastError());
    return MB200_OK;
}

static int run_step(mb200_ctx* ctx, mb200_csc* s, const mb200_seqs* seqs, const int64_t* seq_idx, bool backward) {
    const CscDims d = s->d;
    if (seqs->ragged) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "csc: the network needs sequences of one length; this store has rows of different lengths (a ragged store serves the scan only)");
    if (seqs->Lb != d.Lb) MB_FAIL(ctx, MB200_E_INVALID, "csc: model built for Lb=%d, sequences have Lb=%lld", d.Lb, (long long)seqs->Lb);
    if (seqs->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(seqs)); if (rc) return rc; }
    int64_t* slot = s->idx_pinned + (size_t)(s->ring++ % IDX_RING) * d.NS;
    for (int i = 0; i < d.NS; ++i) {
        if (seq_idx[i] < 0 || seq_idx[i] >= seqs->N) MB_FAIL(ctx, MB200_E_INVALID, "csc: sequence index %lld out of range", (long long)seq_idx[i]);
        slot[i] = seq_idx[i];
    }
    MB_CUDA(ctx, cudaMemcpyAsync(s->idx_dev, slot, (size_t)d.NS * 8, cudaMemcpyHostToDevice, ctx->stream));
    return launch_step(ctx, s, seqs->words, seqs->rowwords, s->idx_dev, backward);
}

// a batch that arrives from the host as ASCII rows: packed to 2 bit/base on the host (NS*Lb bytes, a few hundred), one H2D copy
static int run_step_host(mb200_ctx* ctx, mb200_csc* s, const uint8_t* ascii, int64_t n_rows, bool backward) {
    const CscDims d = s->d;
    if (n_rows != d.NS) MB_FAIL(ctx, MB200_E_INVALID, "csc: expected %d rows (groups x batch_size), got %lld", d.NS, (long long)n_rows);
    const int64_t rw = (d.Lb + 15) / 16;
    uint32_t* slot = s->batch_pinned + (size_t)(s->ring++ % IDX_RING) * d.NS * rw;
    for (int64_t n = 0; n < d.NS; ++n)
        for (int64_t w = 0; w < rw; ++w) {
            uint32_t word = 0;
            for (int i = 0; i < 16 && w * 16 + i < d.Lb; ++i) {
                const uint8_t c = ascii[n * d.Lb + w * 16 + i] & 0xDFu;
                uint32_t code;
                if (c == 'A') code = 0; else if (c == 'C') code = 1; else if (c == 'G') code = 2; else if (c == 'T') code = 3;
                else MB_FAIL(ctx, MB200_E_BAD_SEQUENCE, "csc: row %lld holds a symbol that is not A,C,G,T", (long long)n);
                word |= code << (2 * i);
            }
            slot[n * rw + w] = word;
        }
    MB_CUDA(ctx, cudaMemcpyAsync(s->batch_words, slot, (size_t)d.NS * rw * 4, cudaMemcpyHostToDevice, ctx->stream));
    return launch_step(ctx, s, s->batch_words, rw, s->idx_identity_dev, backward);
}


// The fused reverse pass handles top-q supports of up to FZ_KCAP entries per sequence (q = 32 plus exact ties) and code lists of up to
// LIST_CAP entries.  A step beyond that (ties at the q-th value: an all-zero top-q input, or equal values at many positions of a
// repetitive sequence) raises the error word.  That step is then run again on the same batch, which is still in
// idx_dev or batch_words, through the kernel-per-op tape: its consumers take their dense paths for such lists, so the step returns the
// gradient the reference computes instead of an error.  k_adabelief and k_l1_F read the same word and skip a flagged gradient.
static bool fused_flagged(const mb200_csc* s) { return s->fused_bwd && s->fz_err_host && *s->fz_err_host != 0; }

static int fused_fallback(mb200_ctx* ctx, mb200_csc* s) {
    *s->fz_err_host = 0;
    MB_CUDA(ctx, cudaMemsetAsync(s->fzw.err, 0, 4, ctx->stream));
    MB_CUDA(ctx, cudaMemsetAsync(s->fz_sync, 0, s->fz_zero_bytes, ctx->stream));
    const int64_t c0 = g_lk_count;
    enqueue_step(s, s->last_words, s->last_rowwords, s->last_idx, true, ctx->stream, true);
    ctx->launches[T_CSC] += g_lk_count - c0;
    // the fully fused step expects its d x slots zero when it begins (their reader clears them); the tape leaves the whole arena written
    MB_CUDA(ctx, cudaMemsetAsync(s->grad, 0, (s->arena + s->grad_extra) * 4, ctx->stream));
    MB_CUDA(ctx, cudaGetLastError());
    return MB200_OK;
}

// loss (and gradient) of n_groups batches.  seq_idx: n_groups*batch_size indices into seqs.
// loss_out: n_groups*3 floats {total, reconstruction, syntax} per group; grads: n_trainable floats = mean over groups (or NULL).
extern "C" int32_t mb200_csc_loss_grad(mb200_ctx* ctx, mb200_csc* s, const mb200_seqs* seqs, const int64_t* seq_idx, float* loss_out, float* grads) {
    if (!ctx || !s || !seqs || !seq_idx) return MB200_E_INVALID;
    if (s->xyz_only) MB_FAIL(ctx, MB200_E_INVALID, "csc: handle was created forward_only");
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    mb_reset_timing(ctx);
    MbTimers tm(ctx);
    const int tt = tm.begin(T_TOTAL), tc = tm.begin(T_CSC);
    int rc = run_step(ctx, s, seqs, seq_idx, true);
    if (rc) return rc;
    tm.end(tc);
    const int td = tm.begin(T_D2H);
    if (loss_out) MB_CUDA(ctx, cudaMemcpyAsync(loss_out, s->data + s->loss.off, (size_t)s->d.G * 3 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (grads) MB_CUDA(ctx, cudaMemcpyAsync(grads, s->g_raw, (size_t)s->n_train * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (s->fused_bwd) MB_CUDA(ctx, cudaMemcpyAsync(s->fz_err_host, s->fzw.err, 4, cudaMemcpyDeviceToHost, ctx->stream));
    tm.end(td); tm.end(tt);
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    tm.collect();
    if (fused_flagged(s)) {
        rc = fused_fallback(ctx, s); if (rc) return rc;
        if (loss_out) MB_CUDA(ctx, cudaMemcpyAsync(loss_out, s->data + s->loss.off, (size_t)s->d.G * 3 * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (grads) MB_CUDA(ctx, cudaMemcpyAsync(grads, s->g_raw, (size_t)s->n_train * 4, cudaMemcpyDeviceToHost, ctx->stream));
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return MB200_OK;
}

// forward + reverse pass only; gradients stay on the device (mb200_csc_device_ptrs) so that the host framework can
// all-reduce them in place (one NCCL call) before mb200_csc_adabelief_step.  Asynchronous on the ctx stream.
extern "C" int32_t mb200_csc_step_begin(mb200_ctx* ctx, mb200_csc* s, const mb200_seqs* seqs, const int64_t* seq_idx) {
    if (!ctx || !s || !seqs || !seq_idx) return MB200_E_INVALID;
    if (s->xyz_only) MB_FAIL(ctx, MB200_E_INVALID, "csc: handle was created forward_only");
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    return run_step(ctx, s, seqs, seq_idx, true);
}

// AdaBelief update of the trainable vector with the gradients currently on the device (train.jl:46), then the
// early-stop statistic l1 = sum |prep_syntax_filters(F)| (train.jl:47).  Blocks; returns mean loss of the last step.
// same as mb200_csc_step_begin for a batch handed over as host ASCII rows (n_rows = n_groups*batch_size rows of Lb bytes): the
// reference's `S |> gpu` per step (train.jl:41) with 1 B/bp instead of 16 B/bp.
extern "C" int32_t mb200_csc_step_begin_host(mb200_ctx* ctx, mb200_csc* s, const uint8_t* ascii_rows, int64_t n_rows) {
    if (!ctx || !s || !ascii_rows) return MB200_E_INVALID;
    if (s->xyz_only) MB_FAIL(ctx, MB200_E_INVALID, "csc: handle was created forward_only");
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    return run_step_host(ctx, s, ascii_rows, n_rows, true);
}

extern "C" int32_t mb200_csc_adabelief_step(mb200_ctx* ctx, mb200_csc* s, float eta, float beta1, float beta2, float eps,
                                            float* loss_out, float* l1_F_out) {
    if (!ctx || !s) return MB200_E_INVALID;
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    const unsigned int* err = s->fused_bwd ? s->fzw.err : nullptr;
    // with a communicator the flag is read before the gradient leaves the rank: a flagged step is re-run on the tape first, so every rank
    // still makes exactly one all-reduce per step
    if (err && ctx->comm && ctx->world > 1) {
        MB_CUDA(ctx, cudaMemcpyAsync(s->fz_err_host, err, 4, cudaMemcpyDeviceToHost, ctx->stream));
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (fused_flagged(s)) { const int rc = fused_fallback(ctx, s); if (rc) return rc; }
    }
    // data parallel (SURVEY §8e): ONE all-reduce (average) of the n_train gradients per step, on the stream the reverse pass ran on
    { const int rc = mb_comm_allreduce_f32(ctx, s->g_raw, (size_t)s->n_train, true); if (rc) return rc; }
    const float c1 = 1.f - powf(beta1, (float)(s->step_count + 1)), c2 = 1.f - powf(beta2, (float)(s->step_count + 1));
    float* d_l1 = s->data + s->loss.off + (size_t)s->d.G * 3;       // K slots right after the per-group losses
    for (int attempt = 0; attempt < 2; ++attempt) {
        lk(k_adabelief, nblk(s->n_train, 256), 256, 0, ctx->stream, s->p_raw, (const float*)s->g_raw, s->mt, s->st, eta, beta1, beta2, eps * eps, c1, c2, (int)s->n_train, err);
        // l1(F): one term per syntax filter, summed on the host in a fixed order — bit-identical on every rank, so that all ranks of a
        // data-parallel run take the early-stop branch (train.jl:47-52) on the same step
        lk(k_l1_F, s->d.K, 256, 0, ctx->stream, (const float*)(s->p_raw + s->off_F), d_l1, s->d, err);
        ctx->launches[T_CSC] += 2;
        MB_CUDA(ctx, cudaMemcpyAsync(s->host_out, s->data + s->loss.off, ((size_t)s->d.G * 3 + s->d.K) * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (err) MB_CUDA(ctx, cudaMemcpyAsync(s->fz_err_host, err, 4, cudaMemcpyDeviceToHost, ctx->stream));
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (!fused_flagged(s)) break;
        // one GPU, flagged step: nothing was updated; take the tape's gradient and update once more
        const int rc = fused_fallback(ctx, s); if (rc) return rc;
    }
    s->step_count += 1;
    if (loss_out) { float m = 0.f; for (int g = 0; g < s->d.G; ++g) m += s->host_out[g * 3]; *loss_out = m / (float)s->d.G; }
    if (l1_F_out) { float l1 = 0.f; for (int k = 0; k < s->d.K; ++k) l1 += s->host_out[(size_t)s->d.G * 3 + k]; *l1_F_out = l1; }
    return MB200_OK;
}

// debug / test access to named intermediates of the last forward pass: "z","y","x","zy","D","F","D0","F0","loss"
extern "C" int32_t mb200_csc_get_buffer(mb200_ctx* ctx, mb200_csc* s, const char* name, float* out, int64_t n) {
    if (!ctx || !s || !name || !out) return MB200_E_INVALID;
    auto it = s->named.find(name);
    if (it == s->named.end()) MB_FAIL(ctx, MB200_E_INVALID, "csc: no buffer named %s", name);
    int64_t have = (int64_t)it->second.n;
    if (std::string(name) == "loss") have = (int64_t)s->d.G * 3;
    if (std::string(name) == "D" || std::string(name) == "F") have = (std::string(name) == "D") ? (int64_t)s->d.G * s->d.f_len * s->d.M : (int64_t)s->d.G * s->d.h * s->d.M2 * s->d.K;
    if (n != have) MB_FAIL(ctx, MB200_E_INVALID, "csc: buffer %s has %lld floats", name, (long long)have);
    MB_CUDA(ctx, cudaMemcpyAsync(out, s->data + it->second.off, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
}

// the batch-median mask alone (create_ZY_mask + cat_ZY, model.jl:194-210) on host arrays z,y [G][B*c][M] -> zy [G][B*c][2M], med [G]:
// runs the very kernel the step uses for this handle's shape, so order-statistic corner cases can be checked in isolation
extern "C" int32_t mb200_csc_median_mask(mb200_ctx* ctx, mb200_csc* s, const float* z, const float* y, float* zy_out, float* med_out) {
    if (!ctx || !s || !z || !y || !zy_out || !med_out) return MB200_E_INVALID;
    const CscDims d = s->d;
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t nZ = (size_t)d.NS * d.c * d.M;
    float* buf = nullptr;
    MB_CUDA(ctx, cudaMalloc(&buf, (4 * nZ + d.G) * 4));
    float *dz = buf, *dy = buf + nZ, *dzy = buf + 2 * nZ, *dmed = buf + 4 * nZ;
    cudaMemcpyAsync(dz, z, nZ * 4, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(dy, y, nZ * 4, cudaMemcpyHostToDevice, ctx->stream);
    const bool ms_cluster = s->mask_cap <= MS_MAXV * 512 && d.G < s->ms_cluster_maxg;
    const int ms_cap1 = (int)std::min<int64_t>(2 * (int64_t)d.B * d.c * d.M, 49152);
    if (ms_cluster) lk(k_mask_scale_c, d.G * CL, MS_THREADS, ((size_t)s->mask_cap + 2 * MS_BINS + MS_CAND) * 4, ctx->stream, dz, dy, dzy, dmed, s->mask_cap, d);
    else if (s->batched) lk(k_mask_scale_g, d.G, MG_THREADS, 0, ctx->stream, dz, dy, dzy, dmed, d);
    else lk(k_mask_scale_s, d.G, 1024, (size_t)ms_cap1 * 4, ctx->stream, dz, dy, dzy, dmed, ms_cap1, d);
    cudaMemcpyAsync(zy_out, dzy, 2 * nZ * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(med_out, dmed, (size_t)d.G * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    cudaFree(buf);
    MB_CUDA(ctx, e);
    return MB200_OK;
}

// ---------------------------------------------------------------------------------------------
// code retrieval (inference/_1_code_retrieval.jl:33-56): forward-only ADMM_XYZ over consecutive groups of batch_size
// sequences; non-zeros of X as (position, fil, seq, Float16 mag), ordered by seq, fil, position.
// ---------------------------------------------------------------------------------------------
#define CODE_SLOTS 96          // records per sequence of the first emission; a batch with a longer sequence is emitted again with a wider stride
__global__ void __launch_bounds__(128) k_emit_codes(const float* __restrict__ x, int64_t seq0, mb200_code* __restrict__ slots, int32_t* __restrict__ counts, int stride, CscDims d) {
    PDL_SYNC();
    // one warp per sequence walks (fil, position) in order and compacts entries > 0 with ballots
    const int64_t n = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= d.NS) return;
    const int E = d.l * d.K;
    int cnt = 0;
    for (int e0 = 0; e0 < E; e0 += 32) {
        const int e = e0 + lane;                      // e = fil * l + position
        float v = 0.f; int k = 0, i = 0;
        if (e < E) { k = e / d.l; i = e - k * d.l; v = x[(n * d.l + i) * d.K + k]; }
        const bool hit = v > 0.f;
        const unsigned m = __ballot_sync(FULLMASK, hit);
        if (hit) {
            const int o = cnt + __popc(m & ((1u << lane) - 1u));
            if (o < stride) {
                mb200_code c; c.position = (uint16_t)i; c.fil = (uint16_t)k; c.seq = (uint32_t)(seq0 + n);
                c.mag_f16 = __half_as_ushort(__float2half_rn(v)); c._pad = 0;
                slots[n * stride + o] = c;
            }
        }
        cnt += __popc(m);
    }
    if (lane == 0) counts[n] = cnt;
}

// decodes [first_seq, first_seq + n_seqs); records go to `out` (up to cap) and, when given, are appended to `vec`
static int32_t codes_impl(mb200_ctx* ctx, mb200_csc* s, const mb200_seqs* seqs, int64_t first_seq, int64_t n_seqs,
                          mb200_code* out, int64_t cap, int64_t* n_out, std::vector<mb200_code>* vec) {
    if (!ctx || !s || !seqs || !n_out) return MB200_E_INVALID;
    const CscDims d = s->d;
    if (seqs->ragged) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "csc_codes: code retrieval needs sequences of one length; this store has rows of different lengths (a ragged store serves the scan only)");
    if (seqs->Lb != d.Lb) MB_FAIL(ctx, MB200_E_INVALID, "csc: model built for Lb=%d, sequences have Lb=%lld", d.Lb, (long long)seqs->Lb);
    if (seqs->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(seqs)); if (rc) return rc; }
    if (first_seq < 0 || n_seqs < 0 || first_seq + n_seqs > seqs->N || n_seqs % d.B) MB_FAIL(ctx, MB200_E_INVALID, "csc_codes: range must be whole batches inside the data");
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    mb_reset_timing(ctx);
    MbTimers tm(ctx);
    const int tt = tm.begin(T_TOTAL);
    std::vector<mb200_code> h_slots;
    std::vector<int32_t> h_cnt(d.NS);
    // k_emit_codes on the x of the last forward pass: `stride` records per sequence, then counts and records to the host
    auto emit = [&](int64_t seq0, int stride) -> int {
        const int rc = mb_ensure_buf(ctx, BUF_CODES, (size_t)d.NS * stride * sizeof(mb200_code) + (size_t)d.NS * 4 + 256); if (rc) return rc;
        mb200_code* d_slots = (mb200_code*)ctx->bufs[BUF_CODES];
        int32_t* d_cnt = (int32_t*)(d_slots + (size_t)d.NS * stride);
        lk(k_emit_codes, nblk((int64_t)d.NS * 32, 128), 128, 0, ctx->stream, s->data + s->named["x"].off, seq0, d_slots, d_cnt, stride, d);
        ctx->launches[T_CSC] += 1;
        MB_CUDA(ctx, cudaGetLastError());
        const int td = tm.begin(T_D2H);
        h_slots.resize((size_t)d.NS * stride);
        MB_CUDA(ctx, cudaMemcpyAsync(h_cnt.data(), d_cnt, (size_t)d.NS * 4, cudaMemcpyDeviceToHost, ctx->stream));
        MB_CUDA(ctx, cudaMemcpyAsync(h_slots.data(), d_slots, (size_t)d.NS * stride * sizeof(mb200_code), cudaMemcpyDeviceToHost, ctx->stream));
        tm.end(td);
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return MB200_OK;
    };
    int64_t total = 0; bool overflow = false;
    for (int64_t s0 = 0; s0 < n_seqs; s0 += d.NS) {
        const int64_t ns = std::min<int64_t>(d.NS, n_seqs - s0);
        for (int i = 0; i < d.NS; ++i) s->idx_pinned[i] = first_seq + s0 + (i < ns ? i : 0);   // tail: repeat a valid sequence, results ignored
        MB_CUDA(ctx, cudaMemcpyAsync(s->idx_dev, s->idx_pinned, (size_t)d.NS * 8, cudaMemcpyHostToDevice, ctx->stream));
        const int tc = tm.begin(T_CSC);
        // forward-only: run ops up to the last XYZ pass (a forward_only handle holds exactly those)
        const int64_t c0 = g_lk_count;
        lk(k_unpack_bases, nblk((int64_t)d.NS * d.Lb, 256), 256, 0, ctx->stream, seqs->words, seqs->rowwords, s->idx_dev, s->bases, d);
        for (auto& op : s->tape) { if (op.kind) break; op.fwd(ctx->stream); if (std::string(op.name) == "df_mask") break; }
        ctx->launches[T_CSC] += g_lk_count - c0;
        tm.end(tc);
        int stride = CODE_SLOTS;
        int rc = emit(first_seq + s0, stride); if (rc) return rc;
        const int mx = *std::max_element(h_cnt.begin(), h_cnt.end());      // the tail's repeated sequences count too: they share the stride
        if (mx > stride) { stride = mx; rc = emit(first_seq + s0, stride); if (rc) return rc; }      // x is still in the arena
        for (int64_t i = 0; i < ns; ++i) {
            for (int j = 0; j < h_cnt[i]; ++j) {
                if (vec) vec->push_back(h_slots[(size_t)i * stride + j]);
                else if (total < cap && out) out[total] = h_slots[(size_t)i * stride + j]; else overflow = overflow || (total >= cap);
                ++total;
            }
        }
    }
    tm.end(tt);
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    tm.collect();
    *n_out = total;
    if (!vec && (overflow || (total > cap))) MB_FAIL(ctx, MB200_E_HITS_OVERFLOW, "csc_codes: %lld records, capacity %lld", (long long)total, (long long)cap);
    return MB200_OK;
}

extern "C" int32_t mb200_csc_codes(mb200_ctx* ctx, mb200_csc* s, const mb200_seqs* seqs, int64_t first_seq, int64_t n_seqs,
                                   mb200_code* out, int64_t cap, int64_t* n_out) {
    return codes_impl(ctx, s, seqs, first_seq, n_seqs, out, cap, n_out, nullptr);
}

// Code retrieval sharded over the ranks of the ctx's communicator (SURVEY §8e, third bullet): the batches of batch_size consecutive
// sequences are independent (_1_code_retrieval.jl:38-50), so rank r decodes a contiguous range of whole batches and the records are
// all-gathered in rank order — which is ascending sequence order, i.e. exactly the single-GPU result.  `rank`/`world` < 0: take them
// from the communicator; explicit values with no communicator decode just that shard (no gather; used to test the split on one GPU).
extern "C" int32_t mb200_csc_codes_sharded(mb200_ctx* ctx, mb200_csc* s, const mb200_seqs* seqs, int64_t first_seq, int64_t n_seqs,
                                           int32_t rank, int32_t world, mb200_code* out, int64_t cap, int64_t* n_out) {
    if (!ctx || !s || !seqs || !n_out) return MB200_E_INVALID;
    const bool gather = rank < 0 || world < 0;
    if (gather) { rank = ctx->rank; world = ctx->world; }
    if (world < 1 || rank >= world) MB_FAIL(ctx, MB200_E_INVALID, "csc_codes_sharded: rank %d of %d", rank, world);
    const int B = s->d.B;
    if (n_seqs < 0 || n_seqs % B) MB_FAIL(ctx, MB200_E_INVALID, "csc_codes: range must be whole batches inside the data");
    const int64_t groups = n_seqs / B;
    const int64_t g_lo = groups * rank / world, g_hi = groups * (rank + 1) / world;
    std::vector<mb200_code> mine;
    int64_t n_mine = 0;
    int rc = codes_impl(ctx, s, seqs, first_seq + g_lo * B, (g_hi - g_lo) * B, nullptr, 0, &n_mine, &mine);
    if (rc) return rc;
    if (!gather || world == 1) {
        *n_out = n_mine;
        if (n_mine > cap) MB_FAIL(ctx, MB200_E_HITS_OVERFLOW, "csc_codes: %lld records, capacity %lld", (long long)n_mine, (long long)cap);
        if (n_mine) memcpy(out, mine.data(), (size_t)n_mine * sizeof(mb200_code));
        return MB200_OK;
    }
    std::vector<int64_t> cnt(world, 0);
    rc = mb200_comm_allgather(ctx, &n_mine, cnt.data(), 8); if (rc) return rc;
    int64_t total = 0, mx = 0;
    for (int r = 0; r < world; ++r) { total += cnt[r]; mx = std::max(mx, cnt[r]); }
    *n_out = total;
    // every rank takes part in the gather even when its own `out` is too small (the collective must not dead-lock)
    std::vector<mb200_code> all((size_t)mx * world);
    mine.resize((size_t)mx);
    if (mx) { rc = mb200_comm_allgather(ctx, mine.data(), all.data(), mx * (int64_t)sizeof(mb200_code)); if (rc) return rc; }
    if (total > cap) MB_FAIL(ctx, MB200_E_HITS_OVERFLOW, "csc_codes: %lld records, capacity %lld", (long long)total, (long long)cap);
    int64_t o = 0;
    for (int r = 0; r < world; ++r) { if (cnt[r]) memcpy(out + o, all.data() + (size_t)r * mx, (size_t)cnt[r] * sizeof(mb200_code)); o += cnt[r]; }
    return MB200_OK;
}
