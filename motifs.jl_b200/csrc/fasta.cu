// FASTA -> filtered reads -> train/test split -> k-mer-preserving shuffled backgrounds, in the library (SURVEY §8f-2).
//
// Reference being replaced (paths under the reference's src/loadfasta/):
//   helpers.jl:83-108   reading / read_fasta     drop reads containing N/n, keep at most max_entries, keep reads as long as the
//                                                first one, upper-case
//   helpers.jl:141-159  get_train_test_inds      test size = floor((1 - ratio) n); randperm, sample without replacement, setdiff
//   helpers.jl:206-245  get_data_matrices        seq_shuffle.(reads; k) backgrounds (k = 1 train, k = 2 test: fasta.jl:63),
//                                                est_1st_order_markov_bg
// The reference turns every read into a one-hot Float32 column on the host (16 B/bp, four copies).  Here the reads are uploaded
// once as ASCII, packed to 2 bit/base, and split / shuffled / counted ON THE DEVICE from a host seed; only indices and a 4 + 16
// entry count table travel back.
//
// SeqShuffle 0.2.2 is not vendored in the reference tree [inferred]: `seq_shuffle(s; k)` is taken to be what its name and README
// say, a shuffle that preserves the k-mer counts of s exactly.  For k = 1 that is a uniform permutation; for k >= 2 it is the
// Altschul-Erickson / uShuffle construction: a uniformly random Eulerian walk through the (k-1)-mer graph of s (random
// arborescence towards the last vertex by Wilson's algorithm, remaining out-edges permuted).  The random stream is the
// library's own counter-based generator, so backgrounds are reproducible from (seed, sequence index) on any number of GPUs.
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

struct mb200_fasta { int64_t N = 0, L = 0; std::vector<uint8_t> rows; };

// ---- counter-based random numbers: splitmix64 of (seed, stream, counter) ------------------------------------------------------
__host__ __device__ static inline uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31);
}
__host__ __device__ static inline uint64_t rnd64(uint64_t seed, uint64_t stream, uint64_t ctr) { return mix64(mix64(seed ^ mix64(stream)) + ctr); }
// uniform integer in [0, m), m < 2^32 (multiply-shift; bias < 2^-32)
__host__ __device__ static inline uint32_t rnd_below(uint64_t r, uint32_t m) { return (uint32_t)(((r >> 32) * (uint64_t)m) >> 32); }

// ---- host: FASTA parsing ---------------------------------------------------------------------------------------------------------
extern "C" int32_t mb200_fasta_read(const char* path, int64_t max_entries, mb200_fasta** out, int64_t* N, int64_t* L) {
    if (!path || !out) return MB200_E_INVALID;
    *out = nullptr;
    FILE* fh = fopen(path, "rb");
    if (!fh) return MB200_E_INVALID;
    std::string txt;
    { char buf[1 << 16]; size_t n; while ((n = fread(buf, 1, sizeof buf, fh)) > 0) txt.append(buf, n); }
    fclose(fh);
    // records are split at '>' (helpers.jl:88); the first line of a record is its header, the other lines are joined (:90-91)
    std::vector<std::string> reads;
    size_t pos = 0;
    while (pos <= txt.size()) {
        size_t next = txt.find('>', pos);
        if (next == std::string::npos) next = txt.size();
        if (next > pos) {
            const size_t eol = txt.find('\n', pos);
            std::string read;
            bool has_n = false;
            if (eol != std::string::npos && eol < next)
                for (size_t i = eol + 1; i < next; ++i) { const char c = txt[i]; if (c == '\n') continue; if (c == 'N' || c == 'n') has_n = true; read.push_back(c); }
            if (!has_n) reads.push_back(std::move(read));               // :92
        }
        pos = next + 1;
    }
    if (max_entries >= 0 && (int64_t)reads.size() > max_entries) reads.resize((size_t)max_entries);      // :95
    mb200_fasta* f = new mb200_fasta();
    if (!reads.empty()) {
        f->L = (int64_t)reads[0].size();
        for (auto& r : reads) if ((int64_t)r.size() == f->L) {                                            // :98
            for (char c : r) f->rows.push_back((uint8_t)((c >= 'a' && c <= 'z') ? c - 32 : c));        // uppercase, :107
            ++f->N;
        }
    }
    if (N) *N = f->N;
    if (L) *L = f->L;
    *out = f;
    return MB200_OK;
}
extern "C" int32_t mb200_fasta_rows(const mb200_fasta* f, uint8_t* out_rows) {
    if (!f || !out_rows) return MB200_E_INVALID;
    if (!f->rows.empty()) memcpy(out_rows, f->rows.data(), f->rows.size());
    return MB200_OK;
}
extern "C" int32_t mb200_fasta_free(mb200_fasta* f) { if (!f) return MB200_E_INVALID; delete f; return MB200_OK; }

// ---- host: FASTA records as they are (peak sets, genomes) ---------------------------------------------------------------------
// Every record is kept, whatever its length.  A record's coordinates count every sequence byte (N and IUPAC codes included);
// the maximal runs of A/C/G/T (either case, upper-cased here) are its fragments, the unit the ragged stores hold.
struct mb200_records {
    std::string names;                                   // NUL-terminated names, record order
    std::vector<int64_t> rec_len;
    std::vector<int64_t> frag_rec, frag_start, frag_len;
    std::vector<uint8_t> bases;                          // fragments concatenated
};

extern "C" int32_t mb200_records_read(const char* path, mb200_records** out) {
    if (!path || !out) return MB200_E_INVALID;
    *out = nullptr;
    FILE* fh = fopen(path, "rb");
    if (!fh) return MB200_E_INVALID;
    mb200_records* R = new mb200_records();
    static const uint8_t kUpper[4] = {'A', 'C', 'G', 'T'};
    int64_t pos = 0;                                     // position inside the current record
    bool in_rec = false, header = false, line_start = true, name_done = false, in_frag = false;
    auto close_frag = [&]() { if (in_frag) { R->frag_len.back() = pos - R->frag_start.back(); in_frag = false; } };
    char buf[1 << 16]; size_t got;
    while ((got = fread(buf, 1, sizeof buf, fh)) > 0) {
        for (size_t i = 0; i < got; ++i) {
            const uint8_t c = (uint8_t)buf[i];
            if (c == '\n') { line_start = true; if (header) { header = false; R->names.push_back('\0'); } continue; }
            if (c == '\r') continue;
            if (line_start && c == '>') {                // a new record
                close_frag();
                if (in_rec) R->rec_len.back() = pos;
                R->rec_len.push_back(0); pos = 0;
                in_rec = true; header = true; name_done = false; line_start = false;
                continue;
            }
            line_start = false;
            if (header) {
                if (c == ' ' || c == '\t' || c == '\v' || c == '\f') name_done = true;
                else if (!name_done) R->names.push_back((char)c);
                continue;
            }
            if (!in_rec || c == ' ' || c == '\t') continue;   // text before the first header, blanks inside sequence lines
            const uint8_t u = (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c;
            const int code = u == 'A' ? 0 : u == 'C' ? 1 : u == 'G' ? 2 : u == 'T' ? 3 : -1;
            if (code >= 0) {
                if (!in_frag) { R->frag_rec.push_back((int64_t)R->rec_len.size() - 1); R->frag_start.push_back(pos); R->frag_len.push_back(0); in_frag = true; }
                R->bases.push_back(kUpper[code]);
            } else {
                close_frag();                            // N, IUPAC codes, '-', ...: not scanned
            }
            ++pos;
        }
    }
    const bool err = ferror(fh) != 0;
    fclose(fh);
    if (header) R->names.push_back('\0');
    close_frag();
    if (in_rec) R->rec_len.back() = pos;
    if (err) { delete R; return MB200_E_INVALID; }
    *out = R;
    return MB200_OK;
}
extern "C" int32_t mb200_records_counts(const mb200_records* r, int64_t* n_records, int64_t* n_fragments, int64_t* n_bases, int64_t* name_bytes) {
    if (!r) return MB200_E_INVALID;
    if (n_records) *n_records = (int64_t)r->rec_len.size();
    if (n_fragments) *n_fragments = (int64_t)r->frag_len.size();
    if (n_bases) *n_bases = (int64_t)r->bases.size();
    if (name_bytes) *name_bytes = (int64_t)r->names.size();
    return MB200_OK;
}
extern "C" int32_t mb200_records_names(const mb200_records* r, char* names, int64_t* lengths) {
    if (!r) return MB200_E_INVALID;
    if (names && !r->names.empty()) memcpy(names, r->names.data(), r->names.size());
    if (lengths && !r->rec_len.empty()) memcpy(lengths, r->rec_len.data(), r->rec_len.size() * 8);
    return MB200_OK;
}
extern "C" int32_t mb200_records_fragments(const mb200_records* r, int64_t* record, int64_t* start, int64_t* length, uint8_t* bases) {
    if (!r) return MB200_E_INVALID;
    const size_t nf = r->frag_len.size();
    if (record && nf) memcpy(record, r->frag_rec.data(), nf * 8);
    if (start && nf) memcpy(start, r->frag_start.data(), nf * 8);
    if (length && nf) memcpy(length, r->frag_len.data(), nf * 8);
    if (bases && !r->bases.empty()) memcpy(bases, r->bases.data(), r->bases.size());
    return MB200_OK;
}
extern "C" int32_t mb200_records_free(mb200_records* r) { if (!r) return MB200_E_INVALID; delete r; return MB200_OK; }

// ---- host: train / test indices (get_train_test_inds, helpers.jl:141-159); 0-based --------------------------------------------------
extern "C" int32_t mb200_fasta_split(int64_t n, double train_test_split_ratio, int32_t shuffle, uint64_t seed,
                                     int64_t* train_idx, int64_t* test_idx, int64_t* n_train, int64_t* n_test) {
    if (n < 0 || !train_idx || !test_idx) return MB200_E_INVALID;
    const int64_t nt = (int64_t)std::floor((1.0 - train_test_split_ratio) * (double)n);            // Int(floor((1-ratio)*n)): 99 of 1000
    if (nt < 0 || nt > n) return MB200_E_INVALID;
    std::vector<int64_t> perm((size_t)n);
    for (int64_t i = 0; i < n; ++i) perm[(size_t)i] = i;
    for (int64_t i = n - 1; i > 0; --i) {                                                          // randperm
        const int64_t j = (int64_t)(rnd64(seed, 1, (uint64_t)i) % (uint64_t)(i + 1));
        std::swap(perm[(size_t)i], perm[(size_t)j]);
    }
    std::vector<char> is_test((size_t)n, 0);
    if (shuffle) {                                                                                 // sample(shuffled, nt, replace=false)
        std::vector<int64_t> pool = perm;
        for (int64_t i = 0; i < nt; ++i) {
            const int64_t j = i + (int64_t)(rnd64(seed, 2, (uint64_t)i) % (uint64_t)(n - i));
            std::swap(pool[(size_t)i], pool[(size_t)j]);
            test_idx[i] = pool[(size_t)i]; is_test[(size_t)pool[(size_t)i]] = 1;
        }
    } else {
        for (int64_t i = 0; i < nt; ++i) { test_idx[i] = n - nt + i; is_test[(size_t)(n - nt + i)] = 1; }
    }
    int64_t o = 0;
    for (int64_t i = 0; i < n; ++i) if (!is_test[(size_t)perm[(size_t)i]]) train_idx[o++] = perm[(size_t)i];    // setdiff keeps randperm order
    if (n_train) *n_train = o;
    if (n_test) *n_test = nt;
    return MB200_OK;
}

// ---- device: gather rows, unpack, shuffle, pack, count ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint32_t* __restrict__ src, int64_t rowwords, const int64_t* __restrict__ idx,
                                                          int64_t n, uint32_t* __restrict__ dst) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * rowwords) return;
    const int64_t r = t / rowwords, w = t - r * rowwords;
    dst[t] = src[idx[r] * rowwords + w];
}
// output word w of window r holds bases [start[r] + 16w, +16) of source row row[r]: a window may start at any base, so a word is
// the funnel shift of two source words (the second is read only when the word needs it: it then lies inside the source row).
// Bits past `len` are zero, as in every store.
__global__ void __launch_bounds__(256) windows_kernel(const uint32_t* __restrict__ src, int64_t rowwords, const int64_t* __restrict__ row,
                                                      const int64_t* __restrict__ start, int64_t n, int64_t len, int64_t owords,
                                                      uint32_t* __restrict__ dst) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * owords) return;
    const int64_t r = t / owords, w = t - r * owords;
    const int64_t b0 = start[r] + 16 * w;
    const uint32_t* sp = src + row[r] * rowwords + (b0 >> 4);
    const int o = (int)(b0 & 15);
    const int64_t nb = min((int64_t)16, len - 16 * w);
    uint32_t word = sp[0];
    if (o) word = __funnelshift_r(word, 16 - o < nb ? sp[1] : 0u, 2 * o);
    if (nb < 16) word &= (1u << (2 * nb)) - 1u;
    dst[t] = word;
}
// lens (ragged stores, may be NULL): ASCII output is 0 past a row's length (codes past it are the padding's zeros anyway)
__global__ void __launch_bounds__(256) unpack_codes_kernel(const uint32_t* __restrict__ words, int64_t rowwords, int64_t n, int64_t Lb, int ascii,
                                                           uint8_t* __restrict__ out, const int64_t* __restrict__ lens) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * Lb) return;
    const int64_t r = t / Lb, p = t - r * Lb;
    const uint32_t c = (words[r * rowwords + (p >> 4)] >> ((p & 15) * 2)) & 3u;
    out[t] = ascii ? (lens && p >= lens[r] ? (uint8_t)0 : (uint8_t)"ACGT"[c]) : (uint8_t)c;
}
__global__ void __launch_bounds__(256) pack_codes_kernel(const uint8_t* __restrict__ codes, int64_t n, int64_t Lb, int64_t rowwords, uint32_t* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * rowwords) return;
    const int64_t r = t / rowwords, w = t - r * rowwords;
    const int nb = (int)min((int64_t)16, Lb - w * 16);
    uint32_t word = 0;
    for (int i = 0; i < nb; ++i) word |= (uint32_t)(codes[r * Lb + w * 16 + i] & 3u) << (2 * i);
    out[t] = word;
}

// One thread per sequence.  in/out/edges: [n][Lb] bytes of scratch.  k = 1: Fisher-Yates.  k >= 2 (V = 4^(k-1) <= 64 vertices): random
// Eulerian walk that uses every (k-1)-mer -> base transition of the sequence exactly once (k-mer counts, first and last (k-1)-mer kept).
#define SHUF_MAXV 64
__global__ void __launch_bounds__(128) shuffle_rows_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint8_t* __restrict__ edges,
                                                           int64_t n, int Lb, int k, uint64_t seed, int64_t seq0, const int64_t* __restrict__ lens) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int64_t stride = Lb;
    const uint8_t* s = in + r * stride;
    uint8_t* o = out + r * stride;
    const uint64_t stream = (uint64_t)(seq0 + r);
    uint64_t ctr = 0;
    if (lens) {                                         // ragged store: shuffle this row's own bases; the padding stays zero
        const int Ln = (int)lens[r];
        for (int i = Ln; i < Lb; ++i) o[i] = 0;
        Lb = Ln;
    }
    if (k <= 1 || Lb <= k) {
        for (int i = 0; i < Lb; ++i) o[i] = s[i];
        if (k <= 1)
            for (int i = Lb - 1; i > 0; --i) { const int j = (int)rnd_below(rnd64(seed, stream, ctr++), (uint32_t)(i + 1)); const uint8_t t = o[i]; o[i] = o[j]; o[j] = t; }
        return;
    }
    const int V = 1 << (2 * (k - 1)), E = Lb - k + 1;
    uint8_t* el = edges + r * stride;                     // out-edge lists (the base an edge appends), grouped by source vertex
    int cnt[SHUF_MAXV], off[SHUF_MAXV], nxt[SHUF_MAXV];
    for (int v = 0; v < V; ++v) cnt[v] = 0;
    int v0 = 0;
    for (int i = 0; i < k - 1; ++i) v0 = (v0 << 2) | s[i];
    int u = v0;
    for (int i = 0; i < E; ++i) { ++cnt[u]; u = ((u << 2) | s[i + k - 1]) & (V - 1); }
    const int last = u;
    { int run = 0; for (int v = 0; v < V; ++v) { off[v] = run; run += cnt[v]; cnt[v] = 0; } }
    u = v0;
    for (int i = 0; i < E; ++i) { const int b = s[i + k - 1]; el[off[u] + cnt[u]++] = (uint8_t)b; u = ((u << 2) | b) & (V - 1); }
    // Wilson's algorithm: loop-erased random walks towards `last` choose, per vertex, the edge that is used LAST; uniform over the
    // arborescences (with edge multiplicity), hence a uniform Eulerian walk once the other edges are permuted
    uint64_t in_tree = 1ull << last;
    for (int v = 0; v < V; ++v) {
        if (!cnt[v] || ((in_tree >> v) & 1)) continue;
        int w = v;
        while (!((in_tree >> w) & 1)) { nxt[w] = (int)rnd_below(rnd64(seed, stream, ctr++), (uint32_t)cnt[w]); w = ((w << 2) | el[off[w] + nxt[w]]) & (V - 1); }
        w = v;
        while (!((in_tree >> w) & 1)) { in_tree |= 1ull << w; w = ((w << 2) | el[off[w] + nxt[w]]) & (V - 1); }
    }
    for (int v = 0; v < V; ++v) {
        int m = cnt[v];
        if (!m) continue;
        uint8_t* e = el + off[v];
        if (v != last) { const uint8_t t = e[nxt[v]]; e[nxt[v]] = e[m - 1]; e[m - 1] = t; --m; }      // the exit edge goes last
        for (int i = m - 1; i > 0; --i) { const int j = (int)rnd_below(rnd64(seed, stream, ctr++), (uint32_t)(i + 1)); const uint8_t t = e[i]; e[i] = e[j]; e[j] = t; }
        cnt[v] = 0;                                       // reused as the read cursor below
    }
    for (int i = 0; i < k - 1; ++i) o[i] = s[i];
    u = v0;
    for (int i = 0; i < E; ++i) { const int b = el[off[u] + cnt[u]++]; o[i + k - 1] = (uint8_t)b; u = ((u << 2) | b) & (V - 1); }
}
// chromosome-scale sequences, k = 1: a uniform permutation = sort by random 64-bit keys
__global__ void __launch_bounds__(256) shuffle_keys_kernel(uint64_t* __restrict__ keys, int64_t Lb, uint64_t seed, uint64_t stream) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < Lb) keys[t] = rnd64(seed, stream, (uint64_t)t);
}
__global__ void __launch_bounds__(256) base_counts_kernel(const uint32_t* __restrict__ words, int64_t rowwords, int64_t n, int64_t Lb,
                                                          unsigned long long* __restrict__ out /* 4 + 16 */, const int64_t* __restrict__ lens) {
    __shared__ unsigned long long s_c[20];
    if (threadIdx.x < 20) s_c[threadIdx.x] = 0;
    __syncthreads();
    unsigned int c[20];
    #pragma unroll
    for (int i = 0; i < 20; ++i) c[i] = 0;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n * Lb; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = t / Lb, p = t - r * Lb;
        const int64_t Ln = lens ? lens[r] : Lb;                 // ragged store: only the row's own bases
        if (p >= Ln) continue;
        const uint32_t a = (words[r * rowwords + (p >> 4)] >> ((p & 15) * 2)) & 3u;
        ++c[a];
        if (p + 1 < Ln) { const uint32_t b = (words[r * rowwords + ((p + 1) >> 4)] >> (((p + 1) & 15) * 2)) & 3u; ++c[4 + a * 4 + b]; }
    }
    #pragma unroll
    for (int i = 0; i < 20; ++i) if (c[i]) atomicAdd(&s_c[i], (unsigned long long)c[i]);
    __syncthreads();
    if (threadIdx.x < 20 && s_c[threadIdx.x]) atomicAdd(&out[threadIdx.x], s_c[threadIdx.x]);
}

// rows idx[0..n) of `src` as a new store (train / test sets of one upload: `dna_read[train_set_inds]`, helpers.jl:214-215)
extern "C" int32_t mb200_seqs_gather(mb200_ctx* ctx, const mb200_seqs* src, const int64_t* idx, int64_t n, mb200_seqs** out) {
    if (!ctx || !src || !out || n < 0 || (n > 0 && !idx)) return MB200_E_INVALID;
    *out = nullptr;
    if (src->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(src)); if (rc) return rc; }
    for (int64_t i = 0; i < n; ++i) if (idx[i] < 0 || idx[i] >= src->N) MB_FAIL(ctx, MB200_E_INVALID, "seqs_gather: index %lld out of range", (long long)idx[i]);
    int rc = mb_seqs_alloc(ctx, n, src->Lb, out); if (rc) return rc;
    if (src->ragged) {                                                // the rows keep their lengths (and their zero padding)
        std::vector<int64_t> hl((size_t)n);
        for (int64_t i = 0; i < n; ++i) hl[(size_t)i] = src->hlens[(size_t)idx[i]];
        rc = mb_seqs_set_lens(ctx, *out, std::move(hl));
        if (rc) { mb200_seqs_free(ctx, *out); *out = nullptr; return rc; }
    }
    if (n == 0) return MB200_OK;
    rc = mb_ensure_scratch(ctx, (size_t)n * 8);
    cudaError_t e = cudaSuccess;
    if (!rc) e = cudaMemcpyAsync(ctx->scratch, idx, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (!rc && e == cudaSuccess) {
        const int64_t th = n * src->rowwords;
        gather_rows_kernel<<<(unsigned)((th + 255) / 256), 256, 0, ctx->stream>>>(src->words, src->rowwords, (const int64_t*)ctx->scratch, n, (*out)->words);
        e = cudaStreamSynchronize(ctx->stream);                       // idx is the caller's
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (rc || e != cudaSuccess) { mb200_seqs_free(ctx, *out); *out = nullptr; if (rc) return rc; MB_FAIL(ctx, MB200_E_CUDA, "seqs_gather: %s", cudaGetErrorString(e)); }
    return MB200_OK;
}

// windows [start[i], start[i] + len) of rows row[i] of `src` (fixed or ragged) as a new fixed-length store of n rows of len bases:
// the flanks of best sites (mb200_scan_spacing), or any other fixed-width view of a store without a round trip to the host
extern "C" int32_t mb200_seqs_windows(mb200_ctx* ctx, const mb200_seqs* src, const int64_t* row, const int64_t* start, int64_t n, int64_t len,
                                      mb200_seqs** out) {
    if (!ctx || !src || !out) return MB200_E_INVALID;
    *out = nullptr;
    if (n < 0 || len < 1 || (n > 0 && (!row || !start))) MB_FAIL(ctx, MB200_E_INVALID, "seqs_windows: bad arguments (n=%lld len=%lld)", (long long)n, (long long)len);
    if (src->device != ctx->device) MB_FAIL(ctx, MB200_E_INVALID, "seqs_windows: sequences live on device %d, ctx on %d", src->device, ctx->device);
    for (int64_t i = 0; i < n; ++i) {
        if (row[i] < 0 || row[i] >= src->N) MB_FAIL(ctx, MB200_E_INVALID, "seqs_windows: window %lld: row %lld out of range", (long long)i, (long long)row[i]);
        if (start[i] < 0 || start[i] > mb_row_len(src, row[i]) - len)
            MB_FAIL(ctx, MB200_E_INVALID, "seqs_windows: window %lld: [%lld, %lld) leaves row %lld (%lld bases)", (long long)i, (long long)start[i],
                    (long long)(start[i] + len), (long long)row[i], (long long)mb_row_len(src, row[i]));
    }
    if (src->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(src)); if (rc) return rc; }
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = mb_seqs_alloc(ctx, n, len, out); if (rc) return rc;
    if (n == 0) return MB200_OK;
    rc = mb_ensure_scratch(ctx, (size_t)n * 16);
    cudaError_t e = cudaSuccess;
    if (!rc) e = cudaMemcpyAsync(ctx->scratch, row, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (!rc && e == cudaSuccess) e = cudaMemcpyAsync((int64_t*)ctx->scratch + n, start, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (!rc && e == cudaSuccess) {
        const int64_t th = n * (*out)->rowwords;
        windows_kernel<<<(unsigned)((th + 255) / 256), 256, 0, ctx->stream>>>(src->words, src->rowwords, (const int64_t*)ctx->scratch,
                                                                              (const int64_t*)ctx->scratch + n, n, len, (*out)->rowwords, (*out)->words);
        e = cudaStreamSynchronize(ctx->stream);                       // row / start are the caller's
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (rc || e != cudaSuccess) { mb200_seqs_free(ctx, *out); *out = nullptr; if (rc) return rc; MB_FAIL(ctx, MB200_E_CUDA, "seqs_windows: %s", cudaGetErrorString(e)); }
    return MB200_OK;
}

// seq_shuffle.(reads; k) (helpers.jl:217,221): every sequence of `src` shuffled with its k-mer counts preserved; sequence i of a store
// uses random stream first_stream + i, so that shards of one data set shuffled on different GPUs equal the single-GPU result.
extern "C" int32_t mb200_seqs_shuffle(mb200_ctx* ctx, const mb200_seqs* src, int32_t k, uint64_t seed, int64_t first_stream, mb200_seqs** out) {
    if (!ctx || !src || !out) return MB200_E_INVALID;
    *out = nullptr;
    if (k < 1 || k > 4) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "seqs_shuffle: k = %d (1..4 supported)", k);
    if (src->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(src)); if (rc) return rc; }
    const int64_t n = src->N, Lb = src->Lb;
    const int64_t kShortMax = 65536;
    const bool longseq = Lb > kShortMax;
    bool long_rows = longseq;                                        // some row is longer than kShortMax
    if (src->ragged) { long_rows = false; for (int64_t r = 0; r < n; ++r) long_rows |= src->hlens[(size_t)r] > kShortMax; }
    if (long_rows && k != 1) MB_FAIL(ctx, MB200_E_UNSUPPORTED, "seqs_shuffle: sequences longer than 65536 support k = 1 only");
    int rc = mb_seqs_alloc(ctx, n, Lb, out); if (rc) return rc;
    if (src->ragged) {
        rc = mb_seqs_set_lens(ctx, *out, src->hlens);
        if (rc) { mb200_seqs_free(ctx, *out); *out = nullptr; return rc; }
    }
    if (n == 0) return MB200_OK;
    cudaError_t e = cudaSuccess;
    if (!longseq) {
        const size_t plane = (size_t)n * (size_t)Lb;
        rc = mb_ensure_scratch(ctx, 3 * plane + 256);
        if (!rc) {
            uint8_t* d_in = (uint8_t*)ctx->scratch; uint8_t* d_out = d_in + plane; uint8_t* d_ed = d_out + plane;
            unpack_codes_kernel<<<(unsigned)((plane + 255) / 256), 256, 0, ctx->stream>>>(src->words, src->rowwords, n, Lb, 0, d_in, nullptr);
            shuffle_rows_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(d_in, d_out, d_ed, n, (int)Lb, k, seed, first_stream, src->lens);
            pack_codes_kernel<<<(unsigned)((n * src->rowwords + 255) / 256), 256, 0, ctx->stream>>>(d_out, n, Lb, src->rowwords, (*out)->words);
            e = cudaGetLastError();
        }
    } else {
        // one row at a time.  Rows longer than kShortMax: k = 1 as a sort by random keys.  The short rows of a ragged store take the
        // kernel above (one row per launch), so that a row is shuffled the same way whichever store holds it.
        size_t tmp_bytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint8_t*)nullptr, (uint8_t*)nullptr, (int64_t)Lb, 0, 64, ctx->stream);
        const size_t kb = ((size_t)Lb * 8 + 255) & ~(size_t)255, vb = ((size_t)Lb + 255) & ~(size_t)255;
        const size_t sb = src->ragged ? 3 * (size_t)kShortMax : 0;
        rc = mb_ensure_scratch(ctx, 2 * kb + 2 * vb + tmp_bytes + sb + 512);
        if (!rc) {
            uint8_t* base = (uint8_t*)ctx->scratch;
            uint64_t* k_in = (uint64_t*)base; uint64_t* k_out = (uint64_t*)(base + kb);
            uint8_t* v_in = base + 2 * kb; uint8_t* v_out = v_in + vb; void* tmp = v_out + vb;
            uint8_t* s_in = (uint8_t*)(((uintptr_t)tmp + tmp_bytes + 255) & ~(uintptr_t)255); uint8_t* s_out = s_in + kShortMax; uint8_t* s_ed = s_out + kShortMax;
            for (int64_t r = 0; r < n && e == cudaSuccess; ++r) {
                const int64_t Ln = mb_row_len(src, r);
                uint32_t* dst = (*out)->words + r * src->rowwords;
                if (Ln > kShortMax) {
                    unpack_codes_kernel<<<(unsigned)((Ln + 255) / 256), 256, 0, ctx->stream>>>(src->words + r * src->rowwords, src->rowwords, 1, Ln, 0, v_in, nullptr);
                    shuffle_keys_kernel<<<(unsigned)((Ln + 255) / 256), 256, 0, ctx->stream>>>(k_in, Ln, seed, (uint64_t)(first_stream + r));
                    e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, k_in, k_out, v_in, v_out, (int64_t)Ln, 0, 64, ctx->stream);
                    pack_codes_kernel<<<(unsigned)((src->rowwords + 255) / 256), 256, 0, ctx->stream>>>(v_out, 1, Ln, src->rowwords, dst);
                } else {
                    if (Ln > 0) {
                        unpack_codes_kernel<<<(unsigned)((Ln + 255) / 256), 256, 0, ctx->stream>>>(src->words + r * src->rowwords, src->rowwords, 1, Ln, 0, s_in, nullptr);
                        shuffle_rows_kernel<<<1, 128, 0, ctx->stream>>>(s_in, s_out, s_ed, 1, (int)Ln, k, seed, first_stream + r, nullptr);
                    }
                    pack_codes_kernel<<<(unsigned)((src->rowwords + 255) / 256), 256, 0, ctx->stream>>>(s_out, 1, Ln, src->rowwords, dst);   // zero words past Ln
                }
            }
            if (e == cudaSuccess) e = cudaGetLastError();
        }
    }
    if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (rc || e != cudaSuccess) { mb200_seqs_free(ctx, *out); *out = nullptr; if (rc) return rc; MB_FAIL(ctx, MB200_E_CUDA, "seqs_shuffle: %s", cudaGetErrorString(e)); }
    return MB200_OK;
}

// est_1st_order_markov_bg (helpers.jl:225-226) and get_data_bg (MOTIFs.jl:35-39) need only these: base_counts[4] = occurrences of
// A,C,G,T; transitions[16] = occurrences of base a followed by base b inside a sequence, [a*4 + b].
extern "C" int32_t mb200_seqs_base_counts(mb200_ctx* ctx, const mb200_seqs* seqs, int64_t* base_counts, int64_t* transitions) {
    if (!ctx || !seqs || !base_counts) return MB200_E_INVALID;
    if (seqs->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(seqs)); if (rc) return rc; }
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = mb_ensure_scratch(ctx, 256); if (rc) return rc;
    unsigned long long* d = (unsigned long long*)ctx->scratch;
    MB_CUDA(ctx, cudaMemsetAsync(d, 0, 20 * 8, ctx->stream));
    const int64_t total = seqs->N * seqs->Lb;
    if (total > 0) {
        const unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 8);
        base_counts_kernel<<<grid, 256, 0, ctx->stream>>>(seqs->words, seqs->rowwords, seqs->N, seqs->Lb, d, seqs->lens);
        MB_CUDA(ctx, cudaGetLastError());
    }
    unsigned long long h[20];
    MB_CUDA(ctx, cudaMemcpyAsync(h, d, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 4; ++i) base_counts[i] = (int64_t)h[i];
    if (transitions) for (int i = 0; i < 16; ++i) transitions[i] = (int64_t)h[4 + i];
    return MB200_OK;
}

// the reads back as ASCII rows (N x Lb bytes, "ACGT"): raw_data / raw_data_test of FASTA_DNA, and the oracle's input in the tests
extern "C" int32_t mb200_seqs_to_ascii(mb200_ctx* ctx, const mb200_seqs* seqs, uint8_t* out_rows) {
    if (!ctx || !seqs || !out_rows) return MB200_E_INVALID;
    if (seqs->pending) { const int rc = mb_seqs_finish(ctx, const_cast<mb200_seqs*>(seqs)); if (rc) return rc; }
    MB_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t total = seqs->N * seqs->Lb;
    if (total == 0) return MB200_OK;
    const int64_t chunk_rows = std::max<int64_t>(1, ((int64_t)256 << 20) / seqs->Lb);
    int rc = mb_ensure_scratch(ctx, (size_t)std::min(chunk_rows, seqs->N) * (size_t)seqs->Lb); if (rc) return rc;
    for (int64_t r0 = 0; r0 < seqs->N; r0 += chunk_rows) {
        const int64_t nr = std::min(chunk_rows, seqs->N - r0);
        unpack_codes_kernel<<<(unsigned)((nr * seqs->Lb + 255) / 256), 256, 0, ctx->stream>>>(seqs->words + r0 * seqs->rowwords, seqs->rowwords, nr, seqs->Lb, 1, (uint8_t*)ctx->scratch,
                                                                                             seqs->lens ? seqs->lens + r0 : nullptr);
        MB_CUDA(ctx, cudaGetLastError());
        MB_CUDA(ctx, cudaMemcpyAsync(out_rows + r0 * seqs->Lb, ctx->scratch, (size_t)nr * (size_t)seqs->Lb, cudaMemcpyDeviceToHost, ctx->stream));
        MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return MB200_OK;
}
