/*
 * motifs_b200.h — C ABI of libmotifs_b200.so, the B200 (sm_100a) implementation of the
 * data-parallel hot path of kchu25/MOTIFs.jl.
 *
 * The reference has no FFI: the path sits behind plain Julia functions.  Each entry point below
 * names the reference function (file:line under the reference's src/) whose body it replaces when
 * the Julia host calls this library through `ccall` (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns int32: 0 = MB200_OK, <0 = error; text via mb200_last_error(ctx).
 *   - no exceptions, no torch/C++ types cross the ABI: plain pointers and sizes only.
 *   - the caller owns every host buffer; the library owns device memory behind opaque handles.
 *   - a ctx is bound to one CUDA device and is NOT thread-safe (one in-flight call per ctx).
 *     Calls block until their host-visible outputs are written.
 *   - all indices crossing the ABI are 0-based (the Julia glue adds 1).
 *   - there is no CPU fallback: without a CUDA device mb200_create fails.
 */
#ifndef MOTIFS_B200_H
#define MOTIFS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MB200_OK                 0
#define MB200_E_INVALID         -1   /* bad argument */
#define MB200_E_CUDA            -2   /* CUDA runtime error (see mb200_last_error) */
#define MB200_E_NOMEM           -3
#define MB200_E_BAD_SEQUENCE    -4   /* a byte that is not A,C,G,T (either case) / not one-hot */
#define MB200_E_HITS_OVERFLOW   -5   /* hits_cap too small; *n_hits holds the required size */
#define MB200_E_UNSUPPORTED     -6
#define MB200_E_COMM            -7   /* NCCL missing or a collective failed (see mb200_last_error) */

#define MB200_MAX_MOTIF_LEN     64   /* longest PWM the register-resident scan kernel scores; longer PWMs take a plain kernel */

typedef struct mb200_ctx  mb200_ctx;
typedef struct mb200_seqs mb200_seqs;
typedef struct mb200_csc  mb200_csc;

/* ---- context ------------------------------------------------------------------------------ */
int32_t     mb200_version(void);
int32_t     mb200_create(mb200_ctx** out, int32_t device_id);
int32_t     mb200_destroy(mb200_ctx* ctx);
const char* mb200_last_error(const mb200_ctx* ctx);
/* Launch all kernels of this ctx on an existing stream (a cudaStream_t passed as void*; NULL =
 * the ctx's own stream).  Lets a host that already owns a stream (e.g. torch) order work. */
int32_t     mb200_set_stream(mb200_ctx* ctx, void* cuda_stream);
/* Device-side timing of the last scan/step call, measured with CUDA events on the launch stream.
 * out_ms[0]=pack, [1]=scan kernel, [2]=count kernel, [3]=emit (+prefix), [4]=csc step,
 * [5]=h2d copies, [6]=d2h copies, [7]=total of the call.  launches[i] = kernels launched. */
int32_t     mb200_last_timing(const mb200_ctx* ctx, float* out_ms8, int64_t* launches8);

/* ---- multi-GPU: one process per GPU, one NCCL communicator per ctx -------------------------
 * The reference is single-GPU; SURVEY §8e shards the path over sequences: training averages the
 * filter gradients with ONE all-reduce per step (the loop of train.jl:40-52), a scan sums the per-motif
 * counts once (render.jl:70-85), code retrieval shards whole batches (_1_code_retrieval.jl:38-50).
 * Rank 0 calls mb200_comm_unique_id and hands the 128 bytes to the other processes by whatever
 * means the host has (Julia: Distributed / MPI / a file); every rank then calls mb200_comm_init
 * (collective).  With a communicator:
 *   - mb200_csc_adabelief_step averages the gradients over ranks before the update,
 *   - mb200_csc_broadcast_params makes rank `root`'s parameters and optimiser state everybody's,
 *   - mb200_scan / mb200_scan_hist with MB200_SCAN_REDUCE return counts / histograms summed over ranks,
 *   - mb200_csc_codes_sharded decodes this rank's share of the batches and gathers all records.
 * NCCL is loaded at run time (libnccl.so.2); without it mb200_comm_init returns MB200_E_COMM.   */
#define MB200_COMM_ID_BYTES 128
int32_t mb200_comm_unique_id(uint8_t* id_out /* MB200_COMM_ID_BYTES */);
int32_t mb200_comm_init(mb200_ctx* ctx, const uint8_t* id, int32_t rank, int32_t world);
int32_t mb200_comm_destroy(mb200_ctx* ctx);
int32_t mb200_comm_info(const mb200_ctx* ctx, int32_t* rank, int32_t* world, int32_t* nccl_version);
/* small host-buffer exchanges for the host loop (epoch seed, stop flag, record counts); blocking, collective */
int32_t mb200_comm_broadcast(mb200_ctx* ctx, void* host_buf, int64_t bytes, int32_t root);
int32_t mb200_comm_allreduce_i64(mb200_ctx* ctx, int64_t* host_buf, int64_t n);
int32_t mb200_comm_allgather(mb200_ctx* ctx, const void* host_send, void* host_recv, int64_t bytes_per_rank);

/* ---- sequences: replaces the one-hot Float32 arrays of loadfasta/fasta.jl:13-22 ------------
 * Sequences are stored 2 bit/base (A=0,C=1,G=2,T=3; same row order as helpers.jl:125-128),
 * 16 bases per little-endian uint32, each sequence padded to a whole number of words.        */
/* ascii: N rows of Lb bytes, row-major, upper or lower case. */
int32_t mb200_seqs_from_ascii(mb200_ctx* ctx, const uint8_t* ascii, int64_t N, int64_t Lb,
                              mb200_seqs** out);
/* same, but returns at once: the H2D copies and pack kernels are queued on a copy stream of the ctx in 64 MB chunks, and
 * mb200_scan starts on the first sequences while later chunks are still in flight (every other consumer, and
 * mb200_seqs_wait, first waits for the whole upload).  `ascii` must stay valid — and should be pinned — until the first scan
 * of these sequences or mb200_seqs_wait has returned; that call also reports MB200_E_BAD_SEQUENCE.          */
int32_t mb200_seqs_from_ascii_async(mb200_ctx* ctx, const uint8_t* ascii, int64_t N, int64_t Lb,
                                    mb200_seqs** out);
int32_t mb200_seqs_wait(mb200_ctx* ctx, mb200_seqs* seqs);
/* same as mb200_seqs_from_ascii, but `ascii_dev` is a device pointer on ctx's device (no host copy). */
int32_t mb200_seqs_from_device_ascii(mb200_ctx* ctx, const void* ascii_dev, int64_t N, int64_t Lb,
                                     mb200_seqs** out);
/* onehot: the reference's data_matrix (helpers.jl:123-139, fasta.jl:75): Float32, column-major
 * (4*Lb, N) (the singleton middle dimension is a reshape), exactly one 1 per group of 4. */
int32_t mb200_seqs_from_onehot_f32(mb200_ctx* ctx, const float* onehot, int64_t N, int64_t Lb,
                                   mb200_seqs** out);
/* rows of different lengths (a peak set, the N-free fragments of a genome): row i = ascii[offsets[i], offsets[i+1]), offsets has
 * N+1 non-decreasing entries, empty rows are allowed.  Lb = the longest row (at least 1); shorter rows are padded with zero words
 * and every consumer honours each row's own length: mb200_scan / mb200_scan_hist return exactly what they return for each row
 * on its own (start positions 0 .. L_n - len_k), gather / shuffle / base_counts / to_ascii / count_matrices work on [0, L_n).
 * The CSC entry points (training, code retrieval) need one length and return MB200_E_UNSUPPORTED for such a store.        */
int32_t mb200_seqs_from_ascii_ragged(mb200_ctx* ctx, const uint8_t* ascii, const int64_t* offsets, int64_t N,
                                     mb200_seqs** out);
/* the N row lengths; Lb for every row of a fixed-length store */
int32_t mb200_seqs_lengths(const mb200_seqs* s, int64_t* out);
int32_t mb200_seqs_free(mb200_ctx* ctx, mb200_seqs* s);
int32_t mb200_seqs_shape(const mb200_seqs* s, int64_t* N, int64_t* Lb, int64_t* words_per_seq);
/* copy the packed words back (N * words_per_seq uint32) — used by tests. */
int32_t mb200_seqs_download(mb200_ctx* ctx, const mb200_seqs* s, uint32_t* out_words, int64_t n_words);

/* ---- FASTA -> reads -> train/test split -> shuffled backgrounds (SURVEY §8f-2): replaces reading / read_fasta
 *      (loadfasta/helpers.jl:83-108), get_train_test_inds (:141-159), the seq_shuffle.(...; k) backgrounds and
 *      est_1st_order_markov_bg of get_data_matrices (:206-245), get_data_bg (MOTIFs.jl:35-39).  The one-hot matrices of
 *      fasta.jl:61-101 never exist: reads are uploaded once, split / shuffled / counted on the device.               */
typedef struct mb200_fasta mb200_fasta;
/* parse a FASTA file on the host: records split at '>', lines after the header joined, reads containing N/n dropped, at most
 * max_entries kept (< 0: no cap; the reference uses 100 000), reads whose length differs from the first one dropped, upper-cased. */
int32_t mb200_fasta_read(const char* path, int64_t max_entries, mb200_fasta** out, int64_t* N, int64_t* L);
int32_t mb200_fasta_rows(const mb200_fasta* f, uint8_t* out_rows /* N*L bytes */);
int32_t mb200_fasta_free(mb200_fasta* f);
/* parse a FASTA file keeping everything: no cap, no length or N filter.  '>' at the start of a line opens a record, its name is
 * the header up to the first blank; '\r', blanks and tabs in sequence lines are ignored.  A record's coordinates count every
 * other byte.  A,C,G,T in either case (upper-cased, so soft-masked bases are scanned) form the N-free FRAGMENTS of a record;
 * any other byte (N, IUPAC codes, '-') ends a fragment and is not scanned.                                                   */
typedef struct mb200_records mb200_records;
int32_t mb200_records_read(const char* path, mb200_records** out);
int32_t mb200_records_counts(const mb200_records* r, int64_t* n_records, int64_t* n_fragments, int64_t* n_bases, int64_t* name_bytes);
/* names: name_bytes bytes, the record names in order, each NUL-terminated; lengths: n_records record lengths (either may be NULL) */
int32_t mb200_records_names(const mb200_records* r, char* names, int64_t* lengths);
/* per fragment (n_fragments entries each, 0-based): its record, start inside the record and length; bases: n_bases bytes, the
 * fragments' bases concatenated in fragment order (ready for mb200_seqs_from_ascii_ragged).  Any pointer may be NULL.        */
int32_t mb200_records_fragments(const mb200_records* r, int64_t* record, int64_t* start, int64_t* length, uint8_t* bases);
int32_t mb200_records_free(mb200_records* r);
/* 0-based train / test indices: n_test = floor((1 - ratio) * n); shuffle != 0: randperm, test = sample without replacement,
 * train = the remaining indices in randperm order; shuffle == 0: test = the last n_test indices.  train_idx / test_idx: room for n. */
int32_t mb200_fasta_split(int64_t n, double train_test_split_ratio, int32_t shuffle, uint64_t seed,
                          int64_t* train_idx, int64_t* test_idx, int64_t* n_train, int64_t* n_test);
/* rows idx[0..n) of src as a new store (device gather) */
int32_t mb200_seqs_gather(mb200_ctx* ctx, const mb200_seqs* src, const int64_t* idx, int64_t n, mb200_seqs** out);
/* windows of a store as a new fixed-length store of n rows of len bases (device gather): row i holds bases
 * [start[i], start[i] + len) of row row[i] of src (fixed or ragged; a ragged row's own length is the limit).  A window that leaves
 * its row, an index out of range or len < 1: MB200_E_INVALID.                                                              */
int32_t mb200_seqs_windows(mb200_ctx* ctx, const mb200_seqs* src, const int64_t* row, const int64_t* start, int64_t n, int64_t len,
                           mb200_seqs** out);
/* every sequence shuffled with its k-mer counts preserved exactly (k = 1: uniform permutation; k = 2..4: uniform random Eulerian
 * walk through the (k-1)-mer graph, sequences up to 65 536 bp; k = 1 also for chromosome-scale sequences).  Sequence i draws from
 * random stream first_stream + i of `seed`: shards shuffled on different GPUs equal the single-GPU result.          */
int32_t mb200_seqs_shuffle(mb200_ctx* ctx, const mb200_seqs* src, int32_t k, uint64_t seed, int64_t first_stream, mb200_seqs** out);
/* base_counts[4]: occurrences of A,C,G,T; transitions[16] (may be NULL): base a followed by base b within a sequence, [a*4+b] */
int32_t mb200_seqs_base_counts(mb200_ctx* ctx, const mb200_seqs* seqs, int64_t* base_counts, int64_t* transitions);
/* the stored reads as N rows of Lb ASCII bytes */
int32_t mb200_seqs_to_ascii(mb200_ctx* ctx, const mb200_seqs* seqs, uint8_t* out_rows);

/* ---- PWM scan: replaces greedy_search! + get_pos_scores_arr + gpu_scan
 *      (inference/_h3_1_alignment.jl:18-36, 57-87, 89-99), the threshold filter
 *      filter_position_by_best_thresh! (_s2_filter_pos_w_scores.jl:116-125) and the occurrence
 *      counts get_uniq_pos / union_ranges / get_total_occupied_positions
 *      (_h4_overlap_ratio.jl:5-15, 40-79).                                                   */
typedef struct {
    uint32_t seq;        /* 0-based sequence index                                            */
    uint32_t pos;        /* 0-based start position on the forward strand (reference `l` - 1)  */
    uint16_t motif;      /* 0-based motif index                                               */
    uint16_t score_f16;  /* IEEE binary16 bits; bit-identical to the reference's Float16 sum  */
    uint8_t  comp;       /* 0 = scored with pwm, 1 = scored with reverse(pwm) (use_comp)      */
    uint8_t  _pad[3];
} mb200_hit;             /* 16 bytes */

#define MB200_SCAN_FWD          0x1u   /* score with pwm                 (rc=false pass)      */
#define MB200_SCAN_RC           0x2u   /* score with reverse(pwm)        (rc=true pass)       */
#define MB200_SCAN_WANT_HITS    0x4u
#define MB200_SCAN_WANT_COUNTS  0x8u
#define MB200_SCAN_REDUCE       0x20u  /* counts (and mb200_scan_hist's histogram) are summed over the ranks of the ctx's communicator
                                          before they are returned (one all-reduce per call; hit lists stay per rank)          */
#define MB200_SCAN_NO_TENSOR    0x10u  /* thresholded scans: keep the SIMT kernel (default: tcgen05 pre-filter + exact re-scoring, same hit sets) */

/* pwms_f16 : Float16 bits, Julia column-major (K,4,maxlen) exactly as built at
 *            _h3_1_alignment.jl:66-69 with rc=false (element (k,a,ind) at k + K*(a + 4*ind));
 *            the library derives reverse(pwm) itself.
 * lens     : K motif lengths (Int64, as cu(ms.lens)).
 * thresh_f16: K Float16 bits or NULL.  NULL = reference scan semantics "score > 0";
 *            otherwise a hit needs score > 0 AND score > thresh (scan followed by
 *            filter_position_by_best_thresh!).
 * hits     : sorted by (seq, motif, comp, pos) — per (motif, seq) this is the reference's dict
 *            order (forward hits ascending, then reverse hits ascending; _h3_1:38-52,89-99).
 * counts   : K*4 int64, row k = { n_hits, n_unique_start (get_uniq_pos),
 *            coverage as the reference computes it (union_ranges, last interval dropped when a
 *            (motif,seq) has >= 2 hits: _h4_overlap_ratio.jl:48-56), true union coverage }.  */
int32_t mb200_scan(mb200_ctx* ctx, const mb200_seqs* seqs,
                   const uint16_t* pwms_f16, const int64_t* lens, int32_t K, int32_t maxlen,
                   const uint16_t* thresh_f16, uint32_t flags,
                   mb200_hit* hits, int64_t hits_cap, int64_t* n_hits, int64_t* counts);
/* After mb200_scan returned MB200_E_HITS_OVERFLOW (*n_hits = the size needed) the complete list is held by the library: fetch it
 * here instead of scanning again.  The held list is dropped by the next mb200_scan of the ctx.                        */
int32_t mb200_scan_take_hits(mb200_ctx* ctx, mb200_hit* hits, int64_t hits_cap, int64_t* n_hits);
/* which kernel family the last mb200_scan of this ctx used: 0 = scan_kernel (SIMT), 1 = tcgen05 pre-filter + exact re-scoring
 * (thresholded scans, default), 2 = started on the tensor-core path and fell back to scan_kernel (candidate list overflow). */
int32_t mb200_scan_last_path(const mb200_ctx* ctx);

/* Diagnostic, host arithmetic only (no ctx, no device): the error bound E and pre-filter threshold t' = t - E - eps32 the tensor-core
 * path uses for one (motif, strand) slot, so that its guarantee "Float16 running sum > t  =>  real sum > t'" can be checked exhaustively
 * on the CPU (tests/test_scan_prefilter_cpu.py).  cols_f16: len x 4 Float16 bits, row = PWM column in scoring order, entries {A,C,G,T};
 * col0_f16 (4 values, may be NULL): column 0 of the B operand = entries of column 0 minus t', rounded up.  *possible = 0 when no window
 * can exceed the threshold (the slot is disabled).  MB200_E_UNSUPPORTED for non-finite inputs (those calls use the SIMT kernel).       */
int32_t mb200_scan_prefilter_bound(const uint16_t* cols_f16, int32_t len, uint16_t thresh_f16, double* E, double* t_prefilter,
                                   uint16_t* col0_f16, int32_t* possible);

/* Diagnostic, host arithmetic only: the int8 B operand the tensor-core path multiplies for the same slot.  With f = the real-valued
 * filter (col0_f16 above, then the remaining columns): q[j*4+b] = ceil(2^e f[j][b]) + k[j] (entries that cannot take part in a positive
 * window may be raised further), sum_j k[j] = 0, q in [-128, 127], so the integer window sum is >= 2^e times the real-valued one
 * (tests/test_scan_prefilter_int8_cpu.py).  k: len values, q: len x 4.  e, k and q are left unset when *possible = 0.              */
int32_t mb200_scan_prefilter_int8(const uint16_t* cols_f16, int32_t len, uint16_t thresh_f16, int32_t* e, int32_t* k, int8_t* q,
                                  int32_t* possible);

/* Score histogram of the unthresholded scan (hits = score > 0): hist[k*32768 + b] = number of hits of motif k whose Float16
 * score has the 15-bit pattern b (positive halves order like their bit patterns).  Replaces the hit lists as the input of the
 * threshold sweep in get_best_thresh (inference/_s2_filter_pos_w_scores.jl:99-113) and of get_max_score / get_min_score
 * (:11-36).  flags: MB200_SCAN_FWD | MB200_SCAN_RC.                                              */
int32_t mb200_scan_hist(mb200_ctx* ctx, const mb200_seqs* seqs,
                        const uint16_t* pwms_f16, const int64_t* lens, int32_t K, int32_t maxlen,
                        uint32_t flags, uint32_t* hist);

/* Best site per (sequence, motif): the highest score of every window greedy_search! scores (inference/_h3_1_alignment.jl:18-36),
 * the per-sequence motif feature behind AUC and central-enrichment statistics.  Windows of row n (length L_n) and motif k
 * (length m_k) start at 0 .. L_n - m_k, on the requested strands (MB200_SCAN_FWD: pwm, MB200_SCAN_RC: reverse(pwm)); a window's
 * score has the bits mb200_scan reports for it.  NaN windows are ignored, -Inf is a score.  Ties go to the smaller position, then
 * to the forward strand.  The SIMT scan kernel computes it (no tensor-core path: a best site has no threshold to pre-filter with). */
typedef struct {
    uint32_t pos;        /* 0-based start on the forward strand; UINT32_MAX when found == 0          */
    uint16_t score_f16;  /* Float16 bits, identical to mb200_scan's score of that window            */
    uint8_t  comp;       /* 0 = pwm, 1 = reverse(pwm)                                               */
    uint8_t  found;      /* 0: no window of this motif in the row, or every window is NaN           */
} mb200_best;            /* 8 bytes */
/* best[n*K + k] for every row n of seqs and motif k; flags: MB200_SCAN_FWD | MB200_SCAN_RC only (any other bit, a null best or
 * no strand: MB200_E_INVALID).  Rows are per rank: there is nothing to reduce over a communicator.                          */
int32_t mb200_scan_best(mb200_ctx* ctx, const mb200_seqs* seqs, const uint16_t* pwms_f16, const int64_t* lens,
                        int32_t K, int32_t maxlen, uint32_t flags, mb200_best* best);

/* Secondary-motif spacings around primary sites (SpaMo).  An anchor is a primary motif's site of length len at [start, start + len)
 * of row `row`, on strand comp; its margins are the W = margin bases on either side, [start - W, start) and [start + len,
 * start + len + W), both inside the row.  For every (anchor, secondary k) the best window of k (both strands) in the two margins
 * together is found with the mb200_scan_best rule (ties: lower position, so the left margin, then the forward strand).  It is
 * counted when its score is > 0 and > thresh_f16[k] (NULL: > 0), exactly when mb200_scan would report it as a hit.  A counted
 * window at gap g from the primary (g = start - (s + m_k) on the left, s - (start + len) on the right) goes to
 *   hist[((primary * K + k) * 4 + q) * margin + g],  q = 2 * (comp_k != comp) + downstream,
 * where downstream means the right margin for comp = 0 and the left margin for comp = 1 (0: same strand upstream, 1: same strand
 * downstream, 2: opposite upstream, 3: opposite downstream).  sites (n_anchors * K, may be NULL): the best window of each pair, pos
 * in row coordinates, found = counted (pos = UINT32_MAX when the margins hold no window).  The histogram is summed on the device.
 * MB200_E_INVALID: margin outside [1, 65536], n_primary outside [1, 65535], an anchor's primary >= n_primary, comp > 1, len < 1 or
 * a flank leaving its row, a null hist.  MB200_E_NOMEM: the histogram does not fit on the device.                            */
typedef struct {
    int64_t  row;        /* row of seqs                                                              */
    int64_t  start;      /* 0-based start of the primary site in the row                            */
    int32_t  len;        /* primary motif length m_p                                                 */
    uint16_t primary;    /* 0-based primary motif index (< n_primary)                                */
    uint8_t  comp;       /* strand of the primary site: 0 = pwm, 1 = reverse(pwm)                   */
    uint8_t  _pad;
} mb200_anchor;          /* 24 bytes */
int32_t mb200_scan_spacing(mb200_ctx* ctx, const mb200_seqs* seqs, const mb200_anchor* anchors, int64_t n_anchors,
                           int32_t n_primary, int32_t margin, const uint16_t* pwms_f16, const int64_t* lens, int32_t K,
                           int32_t maxlen, const uint16_t* thresh_f16, uint32_t* hist, mb200_best* sites);

/* ---- unrolled convolutional-sparse-coding network: replaces the GPU work inside
 *      forward_pass_return_loss (model.jl:375-395) + gradient(ps) + Flux.Optimise.update!
 *      (train.jl:42-46) and code_retrieval (inference/_1_code_retrieval.jl:33-56).            */
typedef struct {                 /* Hyperparam, model.jl:1-14 (same defaults expected)         */
    int32_t filter_len, M, h, K, q, batch_size, num_pass_xyz, num_pass_df;
    float   magnifying_factor, gamma;
} mb200_hparams;

/* n_groups independent batches of batch_size sequences are processed per call (1 = the reference's
 * step).  forward_only != 0 builds only ADMM_XYZ (enough for mb200_csc_codes, far less memory);
 * forward_only == 2 additionally routes the dense syntax-filter contraction (model.jl:214,251) through
 * the tcgen05/TMEM tensor-core kernel with BF16 operands and FP32 accumulation — NOT bit-comparable
 * with the fp32 path (stated tolerance in tests/test_csc_gpu.py), off by default.                  */
#define MB200_CSC_NO_FUSED 0x100  /* OR into forward_only: keep the kernel-per-op tape instead of the fused persistent forward kernel
                                     (same results within fp32 summation order; for A/B measurements and tests)            */
#define MB200_CSC_NO_FUSED_DF 0x200 /* OR into forward_only: the reverse pass of the loss and the ADMM_DF passes stays on the tape
                                     (the forward kernel and the fused reverse pass of the ADMM_XYZ passes are kept)       */
int32_t mb200_csc_create(mb200_ctx* ctx, const mb200_hparams* hp, int64_t Lb, int32_t n_groups,
                         int32_t forward_only, mb200_csc** out);
int32_t mb200_csc_destroy(mb200_ctx* ctx, mb200_csc* csc);
int32_t mb200_csc_n_params(const mb200_csc* csc, int64_t* n_trainable, int64_t* n_total);
/* flat Float32 parameter vector in Flux.params(cdl) order (model.jl:67-137, arrays only):
 * lambda_sparsity[6] kappa_sparsity[3] lambda_stepsize[6] omega_stepsize[6] kappa_stepsize[3]
 * D[32*M] (Julia (32,1,M) memory order) F[h*2M*K] (Julia (h,2M,1,K) memory order) penalty_xyz[6] mu[3]
 * = n_trainable, followed by the three non-trainable warm-up scalars lambda_sparsity_warmup,
 * lambda_stepsize_warmup, omega_stepsize_warmup (model.jl:68,72-73) = n_total.                  */
int32_t mb200_csc_set_params(mb200_ctx* ctx, mb200_csc* csc, const float* p, int64_t n_total);
int32_t mb200_csc_get_params(mb200_ctx* ctx, mb200_csc* csc, float* p, int64_t n_total);
int32_t mb200_csc_reset_optimizer(mb200_ctx* ctx, mb200_csc* csc);
/* the n_trainable gradients currently on the device (local after step_begin, rank-averaged after adabelief_step) */
int32_t mb200_csc_get_grads(mb200_ctx* ctx, mb200_csc* csc, float* g, int64_t n_trainable);
/* device addresses of the parameter and gradient vectors (n_total floats each), so that the host
 * framework can all-reduce gradients in place with one NCCL call per step.                      */
int32_t mb200_csc_device_ptrs(const mb200_csc* csc, void** params_dev, void** grads_dev);
/* data-parallel start: rank `root`'s parameters, AdaBelief state and step counter replace every rank's (collective; no-op
 * without a communicator).                                                                        */
int32_t mb200_csc_broadcast_params(mb200_ctx* ctx, mb200_csc* csc, int32_t root);
/* loss and gradient of n_groups batches: seq_idx[n_groups*batch_size] indexes `seqs`.
 * loss_out: n_groups*3 floats {loss, reconstruction term, syntax term}; grads: n_trainable floats,
 * mean over groups (NULL to leave them on the device).                                          */
int32_t mb200_csc_loss_grad(mb200_ctx* ctx, mb200_csc* csc, const mb200_seqs* seqs,
                            const int64_t* seq_idx, float* loss_out, float* grads);
/* same computation, asynchronous, results stay on the device */
int32_t mb200_csc_step_begin(mb200_ctx* ctx, mb200_csc* csc, const mb200_seqs* seqs, const int64_t* seq_idx);
/* same for a batch handed over as host ASCII rows (n_groups*batch_size rows of Lb bytes): the per-step `S |> gpu` of train.jl:41 */
int32_t mb200_csc_step_begin_host(mb200_ctx* ctx, mb200_csc* csc, const uint8_t* ascii_rows, int64_t n_rows);
/* AdaBelief update (Flux.Optimise.AdaBelief defaults eta=1e-3, beta=(0.9,0.999), eps=1e-8) with the
 * gradients on the device — averaged over the ranks of the ctx's communicator first (ONE all-reduce of
 * n_trainable floats per step) when there is one; returns the mean loss of that step and l1 = sum|prep_syntax_filters(F)|
 * (the early-stop statistic of train.jl:47-52).                                                  */
int32_t mb200_csc_adabelief_step(mb200_ctx* ctx, mb200_csc* csc, float eta, float beta1, float beta2,
                                 float eps, float* loss_out, float* l1_F_out);
/* named intermediates of the last forward pass ("z","y","x","zy","D","F","D0","F0","loss") — tests */
int32_t mb200_csc_get_buffer(mb200_ctx* ctx, mb200_csc* csc, const char* name, float* out, int64_t n);
/* the batch-median mask alone: cat_ZY + create_ZY_mask, model.jl:194-210.  z,y host [G][B*c][M] (the position-space rows of
 * Z,Y for the handle's shape) -> zy_out [G][B*c][2M] = magnifying_factor * (ZY >= median(ZY[ZY>0])) .* ZY, med_out [G]
 * (-inf when a group has no positive entry).  Same kernel as inside the step.                              */
int32_t mb200_csc_median_mask(mb200_ctx* ctx, mb200_csc* csc, const float* z, const float* y, float* zy_out, float* med_out);

typedef struct {                 /* stored_code_component_t, inference/_0_const.jl:3-4 (0-based) */
    uint16_t position, fil;
    uint32_t seq;
    uint16_t mag_f16, _pad;
} mb200_code;                    /* 12 bytes */
/* ADMM_XYZ forward over sequences first_seq .. first_seq+n_seqs-1 (n_seqs a multiple of batch_size, groups of
 * batch_size consecutive sequences share the median mask like the reference's DataLoader(shuffle=false)).
 * Records ordered by seq, fil, position.                                                        */
int32_t mb200_csc_codes(mb200_ctx* ctx, mb200_csc* csc, const mb200_seqs* seqs, int64_t first_seq,
                        int64_t n_seqs, mb200_code* out, int64_t cap, int64_t* n_out);

/* the same, sharded over the ranks of the ctx's communicator (mb200_comm_init): rank r decodes a contiguous range of whole
 * batches, the records are all-gathered in rank order = ascending sequence order, so every rank receives exactly what a
 * single-GPU mb200_csc_codes returns.  rank = world = -1 takes them from the communicator; explicit (rank, world) decode just
 * that shard without any communication.  Every rank must hold the same `seqs`.                                 */
int32_t mb200_csc_codes_sharded(mb200_ctx* ctx, mb200_csc* csc, const mb200_seqs* seqs, int64_t first_seq, int64_t n_seqs,
                                int32_t rank, int32_t world, mb200_code* out, int64_t cap, int64_t* n_out);

/* ---- positions -> count matrices: replaces posdicts2countmats / msa_add! (inference/_h6_positions2countmat.jl:7-54),
 *      obtain_count_matrices (_3_make_pfms.jl:28-46) and the counting half of enriched_keys2motifs
 *      (_s1_make_motifs.jl:234-259).                                                              */
typedef struct { uint32_t motif, seq, pos, comp; } mb200_site;   /* 0-based; comp != 0 adds the reverse complement */
/* counts: K*maxlen*4 uint32, entry [(k*maxlen + col)*4 + base]; columns >= lens[k] stay 0. */
int32_t mb200_count_matrices(mb200_ctx* ctx, const mb200_seqs* seqs, const mb200_site* sites, int64_t n_sites,
                             const int64_t* lens, int32_t K, int32_t maxlen, uint32_t* counts);

/* ---- score threshold from a p-value: replaces pvalue2score (inference/_h2_Touzet.jl:170-187, with min_score_range, round_pwm,
 *      best_score / worst_score, create_Q, find_largest_alpha :1-168).  Host-side Float64 DP, bit-identical to the reference's
 *      order of additions.  pwm: 4 x m row-major (row = base A,C,G,T); bg: 4 background frequencies; eps: granularity (1e-1 in
 *      _0_const.jl).  *found = 0 when no score qualifies (the reference returns `nothing`).                  */
int32_t mb200_pvalue2score(mb200_ctx* ctx, const double* pwm, int32_t m, double pval, double eps, const double* bg,
                           double* score, int32_t* found);

/* ---- exact p-values of the scan's score: new; the exact p-value of greedy_search!'s Float16 score (_h3_1_alignment.jl:18-36).
 *      A window's score is a sequential Float16 sum, so after every column it is one of the 63 489 non-NaN Float16 values (-0 = +0).
 *      Under a background of independent bases with frequencies bg (A,C,G,T), the survival function S(t) = P(score >= t) of every
 *      (motif, strand) slot is computed exactly over those values on the device, in float64, column by column (DESIGN.md §3.1c).  The
 *      table is the scan's own effective table (the Inf * 0 = NaN rule) and, for comp = 1, that of reverse(pwm).  NaN windows carry no
 *      mass: S(-Inf) is the probability that a window is not NaN.  Two builds of one input are bit-identical.                     */
typedef struct mb200_pvtab mb200_pvtab;
/* pwms_f16, lens, K, maxlen: exactly as for mb200_scan.  The tables take 2K x 63 489 float64 (0.5 MB per slot) of device memory
 * and the build at most 1 GiB more of working space.  MB200_E_INVALID: a null pointer, K < 1, a len outside [1, maxlen], a bg entry
 * that is negative or non-finite, or a bg whose sum is not within 1e-6 of 1.  MB200_E_NOMEM: the tables do not fit.          */
int32_t mb200_pvtab_create(mb200_ctx* ctx, const uint16_t* pwms_f16, const int64_t* lens, int32_t K, int32_t maxlen,
                           const double* bg, mb200_pvtab** out);
int32_t mb200_pvtab_destroy(mb200_ctx* ctx, mb200_pvtab* t);
/* per slot and pval[k] in [0, 1]: s* = the smallest non-NaN value with S(s*) <= pval[k], thresh_f16[k*2 + comp] = the Float16 value
 * just below s*, so that score > thresh <=> S(score) <= pval[k] for every non-NaN score; -Inf when s* = -Inf, +Inf when no value
 * qualifies (pval[k] < S(+Inf)).  A scan at this threshold still needs score > 0.  MB200_E_INVALID: a p outside [0, 1].      */
int32_t mb200_pvtab_thresholds(mb200_ctx* ctx, const mb200_pvtab* t, const double* pval, uint16_t* thresh_f16);
/* p[i] = S(score_f16[i]) of slot (motif[i], comp[i]), gathered on the device; NaN for a NaN score, -0 is looked up as +0.
 * MB200_E_INVALID: a motif >= K or a comp > 1.                                                                                */
int32_t mb200_pvtab_lookup(mb200_ctx* ctx, const mb200_pvtab* t, const uint16_t* motif, const uint8_t* comp,
                           const uint16_t* score_f16, int64_t n, double* p);
/* the whole table of slot (k, comp): out[65536] indexed by Float16 bit pattern, NaN for the NaN patterns. */
int32_t mb200_pvtab_survival(mb200_ctx* ctx, const mb200_pvtab* t, int32_t k, int32_t comp, double* out);

/* ---- code components -> triplet dictionary: replaces get_scanning_range_of_filtered_code_components, enumerate_triplets /
 *      insert_H! (inference/_2_enumerate.jl:25-65) and the key counting of get_words / get_enriched_keys
 *      (inference/_3_make_pfms.jl:3-26).  A key is f1 | f2<<8 | f3<<16 | d12<<24 | d13<<40 with 1-based filter ids (the fields of
 *      the reference's NamedTuple key).  The dictionary itself stays on the device; the host asks for the keys above a count and
 *      then for the values of the keys it selected.                                                   */
typedef struct mb200_triplets mb200_triplets;
typedef struct { uint64_t key; uint32_t count, reserved; uint64_t first; } mb200_key_count;   /* first = rank of the key's first insertion */
typedef struct { uint32_t key_index, range_index, position, reserved; uint64_t order; } mb200_triplet_value;
/* position/fil/seq: the filtered stored_code_components in the order code retrieval returns them (0-based fields, seq
 * ascending).  Builds the sequence ranges exactly like _2_enumerate.jl:25-35 (a range closes when seq != cur_seq, cur_seq counts
 * up by one per closed range, the last range is never closed), sorts every range by position (stable) and counts every
 * triplet's key.  n_ranges / n_triplets may be NULL.                                                    */
int32_t mb200_triplets_create(mb200_ctx* ctx, const uint16_t* position, const uint16_t* fil, const uint32_t* seq, int64_t n_codes,
                              mb200_triplets** out, int64_t* n_ranges, int64_t* n_triplets);
int32_t mb200_triplets_destroy(mb200_ctx* ctx, mb200_triplets* t);
/* the ranges as 0-based half-open [start, stop) index pairs into the code arrays (n_ranges entries each) */
int32_t mb200_triplets_ranges(mb200_ctx* ctx, const mb200_triplets* t, int32_t* start, int32_t* stop);
/* keys with more than min_count values, in no particular order, each with its count and the rank of its first insertion
 * (ascending `first` = the reference Dictionary's iteration order).  *n = how many there are; at most cap are written. */
int32_t mb200_triplets_frequent(mb200_ctx* ctx, mb200_triplets* t, uint32_t min_count, mb200_key_count* out, int64_t cap, int64_t* n);
/* the dictionary values of `keys` (a subset of the last mb200_triplets_frequent result): one record per value with
 * key_index = index into keys, range_index = 1-based index of the sequence range (what insert_H! stores as seq_num),
 * position = 1-based position of the triplet's first component; ascending `order` within a key = insertion order.
 * *n = how many records there are; at most cap are written.                                             */
int32_t mb200_triplets_values(mb200_ctx* ctx, mb200_triplets* t, const uint64_t* keys, int64_t n_keys, mb200_triplet_value* out,
                              int64_t cap, int64_t* n);

#ifdef __cplusplus
}
#endif
#endif /* MOTIFS_B200_H */
