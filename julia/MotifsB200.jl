# MotifsB200.jl — the `ccall` glue a MOTIFs.jl maintainer adds to route the hot path through libmotifs_b200.so.
# Julia is not installed in the build image, so this file is exercised only by inspection; the same symbols are bound and
# tested from Python (motifs.jl_b200/_lib.py, tests/test_abi.py).  Each function replaces the BODY of the reference function
# named in its comment; signatures and return conventions (1-based, Dict{Int,Vector}) stay the reference's.
module MotifsB200

const lib = get(ENV, "MOTIFS_B200_LIB", "libmotifs_b200.so")

struct Hit            # mb200_hit (16 bytes)
    seq::UInt32; pos::UInt32; motif::UInt16; score::Float16; comp::UInt8; p1::UInt8; p2::UInt8; p3::UInt8
end
struct Best           # mb200_best (8 bytes)
    pos::UInt32; score::Float16; comp::UInt8; found::UInt8
end
struct Code           # mb200_code (12 bytes)
    position::UInt16; fil::UInt16; seq::UInt32; mag::Float16; pad::UInt16
end
struct HParams        # mb200_hparams = Hyperparam (model.jl:1-14)
    filter_len::Int32; M::Int32; h::Int32; K::Int32; q::Int32; batch_size::Int32; num_pass_xyz::Int32; num_pass_df::Int32
    magnifying_factor::Float32; gamma::Float32
end

const SCAN_FWD, SCAN_RC, SCAN_WANT_HITS, SCAN_WANT_COUNTS = UInt32(1), UInt32(2), UInt32(4), UInt32(8)
const SCAN_REDUCE = UInt32(32)         # counts / histograms summed over the ranks of the ctx's communicator inside the call
const SCAN_NO_TENSOR = UInt32(16)      # thresholded scans: keep the SIMT kernel (default: tcgen05 pre-filter + exact re-scoring, same hit sets)
scan_last_path(ctx) = ccall((:mb200_scan_last_path, lib), Int32, (Ptr{Cvoid},), ctx)   # 0 SIMT, 1 tensor-core path, 2 fell back

check(ctx, rc) = rc == 0 || error("libmotifs_b200 ($rc): " * unsafe_string(ccall((:mb200_last_error, lib), Cstring, (Ptr{Cvoid},), ctx)))

function create(device::Integer=0)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:mb200_create, lib), Int32, (Ref{Ptr{Cvoid}}, Int32), h, device)
    rc == 0 || error("mb200_create failed ($rc): no B200-class CUDA device")
    h[]
end
destroy(ctx) = ccall((:mb200_destroy, lib), Int32, (Ptr{Cvoid},), ctx)

# replaces the per-batch `cu(float_type_retrieval.(data_matrix[:,1,n:nend]))` uploads (inference/_h3_1_alignment.jl:74) and
# `S |> gpu` (train.jl:41): the whole one-hot array is packed to 2 bit/base once.  data_matrix is (4L,1,N) or (4L,N) Float32.
function upload_onehot(ctx, data_matrix::Array{Float32})
    L4 = size(data_matrix, 1); N = size(data_matrix, ndims(data_matrix))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve data_matrix check(ctx, ccall((:mb200_seqs_from_onehot_f32, lib), Int32,
        (Ptr{Cvoid}, Ptr{Float32}, Int64, Int64, Ref{Ptr{Cvoid}}), ctx, data_matrix, N, L4 ÷ 4, h))
    h[]
end
free_seqs(ctx, s) = ccall((:mb200_seqs_free, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ctx, s)
# raw reads (N rows of L ASCII bytes, as read_fasta leaves them after uppercase.(...)): no one-hot detour.  async=true returns at once;
# keep `ascii` alive (GC.@preserve) until the first gpu_scan of these sequences or wait_seqs has returned.
function upload_ascii(ctx, ascii::Matrix{UInt8}; async=false)          # size(ascii) == (L, N): one column per read
    h = Ref{Ptr{Cvoid}}(C_NULL); L, N = size(ascii)
    rc = async ? ccall((:mb200_seqs_from_ascii_async, lib), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int64, Int64, Ref{Ptr{Cvoid}}), ctx, ascii, N, L, h) :
                 ccall((:mb200_seqs_from_ascii, lib), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int64, Int64, Ref{Ptr{Cvoid}}), ctx, ascii, N, L, h)
    check(ctx, rc); h[]
end
wait_seqs(ctx, s) = check(ctx, ccall((:mb200_seqs_wait, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ctx, s))

# FASTA files as they are (not in the reference, which keeps only equal-length N-free reads): every record, its N-free fragments.
# Like the rest of this file it is untested here (no Julia in the build image); the Python mirror is records.py.
function read_records(path::AbstractString)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    ccall((:mb200_records_read, lib), Int32, (Cstring, Ref{Ptr{Cvoid}}), path, h) == 0 || error("mb200_records_read($path) failed")
    nr, nf, nb, nn = Ref{Int64}(0), Ref{Int64}(0), Ref{Int64}(0), Ref{Int64}(0)
    ccall((:mb200_records_counts, lib), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ref{Int64}, Ref{Int64}), h[], nr, nf, nb, nn)
    names = Vector{UInt8}(undef, nn[]); lengths = Vector{Int64}(undef, nr[])
    ccall((:mb200_records_names, lib), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Ptr{Int64}), h[], names, lengths)
    rec, start, len = Vector{Int64}(undef, nf[]), Vector{Int64}(undef, nf[]), Vector{Int64}(undef, nf[])
    bases = Vector{UInt8}(undef, nb[])
    ccall((:mb200_records_fragments, lib), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{UInt8}), h[], rec, start, len, bases)
    ccall((:mb200_records_free, lib), Int32, (Ptr{Cvoid},), h[])
    name_list = String.(split(String(names), '\0'; keepempty=true))[1:nr[]]
    (names=name_list, lengths=lengths, frag_record=rec, frag_start=start, frag_len=len, bases=bases)   # 0-based record / start
end
# the bucketing rule of INTEGRATION.md: fragments >= minlen, longest first, padding <= 1/8 of the positions of each store
function bucket_fragments(frag_len::Vector{Int64}, minlen::Integer)
    order = sort(findall(>=(minlen), frag_len); by=i -> (-frag_len[i], i))
    buckets = Vector{Vector{Int}}(); i = 1
    while i <= length(order)
        lmax = frag_len[order[i]]; tot = lmax; j = i + 1
        while j <= length(order) && 8 * (tot + frag_len[order[j]]) >= 7 * (j - i + 1) * lmax
            tot += frag_len[order[j]]; j += 1
        end
        push!(buckets, order[i:j-1]); i = j
    end
    buckets
end
# rows of different lengths: offsets (N+1, 0-based, non-decreasing) into the concatenated bytes
function upload_ragged(ctx, ascii::Vector{UInt8}, offsets::Vector{Int64})
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:mb200_seqs_from_ascii_ragged, lib), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Ptr{Int64}, Int64, Ref{Ptr{Cvoid}}),
                     ctx, ascii, offsets, length(offsets) - 1, h))
    h[]
end
function seqs_lengths(s, N::Integer)
    out = Vector{Int64}(undef, N)
    ccall((:mb200_seqs_lengths, lib), Int32, (Ptr{Cvoid}, Ptr{Int64}), s, out) == 0 || error("mb200_seqs_lengths failed")
    out
end

# replaces get_pos_scores_arr + gpu_scan (inference/_h3_1_alignment.jl:57-99).  `pwms` is the (K,4,maxlen) Float16 array the
# reference builds at :65-69 with rc=false; thresh === nothing gives the reference's "score > 0" scan.
function gpu_scan(ctx, seqs, pwms::Array{Float16,3}, lens::Vector{Int64}; thresh::Union{Nothing,Vector{Float16}}=nothing,
                  want_hits=true, reduce=false)
    K, _, maxlen = size(pwms)
    counts = zeros(Int64, 4, K)                       # column k = (n_hits, unique starts, union_ranges coverage, true coverage)
    nhits = Ref{Int64}(0)
    flags = SCAN_FWD | SCAN_RC | SCAN_WANT_COUNTS | (want_hits ? SCAN_WANT_HITS : UInt32(0))
    cap = 1 << 16
    hits = Vector{Hit}(undef, want_hits ? cap : 0)
    thr = thresh === nothing ? Float16[] : thresh      # kept alive (and unmoved) by GC.@preserve below
    while true
        # pointer(hits) is re-evaluated on every iteration: resize! below may move the buffer
        rc = GC.@preserve pwms lens hits counts thr ccall((:mb200_scan, lib), Int32,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float16}, Ptr{Int64}, Int32, Int32, Ptr{Float16}, UInt32, Ptr{Hit}, Int64, Ref{Int64}, Ptr{Int64}),
            ctx, seqs, pwms, lens, K, maxlen, thresh === nothing ? Ptr{Float16}(C_NULL) : pointer(thr), flags | (reduce ? SCAN_REDUCE : UInt32(0)),
            want_hits ? pointer(hits) : Ptr{Hit}(C_NULL), want_hits ? cap : 0, nhits, counts)
        if rc == -5 && want_hits                      # MB200_E_HITS_OVERFLOW: the library holds the complete list, nhits[] is its size
            resize!(hits, nhits[])
            rc = GC.@preserve hits ccall((:mb200_scan_take_hits, lib), Int32, (Ptr{Cvoid}, Ptr{Hit}, Int64, Ref{Int64}), ctx, hits, length(hits), nhits)
        end
        check(ctx, rc); break
    end
    resize!(hits, want_hits ? nhits[] : 0)
    # modify_w_found! (:38-52): hits arrive sorted (seq, motif, comp, pos) => per (motif, seq) forward hits then rc hits
    positions = [Dict{Int,Vector{Int}}() for _ = 1:K]; scores = [Dict{Int,Vector{Float16}}() for _ = 1:K]
    use_comp = [Dict{Int,Vector{Bool}}() for _ = 1:K]
    for h in hits
        m, n = Int(h.motif) + 1, Int(h.seq) + 1
        push!(get!(positions[m], n, Int[]), Int(h.pos) + 1)
        push!(get!(scores[m], n, Float16[]), h.score)
        push!(get!(use_comp[m], n, Bool[]), h.comp != 0)
    end
    positions, scores, use_comp, counts
end

# replaces the loop body of train_ucdl (train.jl:40-52): gradient(ps) do forward_pass_return_loss(...) end ; update! ; l1 test
# fused = false / fused_df = false keep the kernel-per-op tape for the whole step / for the reverse pass of the loss and the ADMM_DF passes
# (MB200_CSC_NO_FUSED = 0x100, MB200_CSC_NO_FUSED_DF = 0x200: A/B measurements and cross-checks; same results within fp32 summation order)
function csc_create(ctx, hp::HParams, L::Integer; n_groups=1, forward_only=false, tensor_cores=false, fused=true, fused_df=true)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    flags = Int32((tensor_cores ? 2 : (forward_only ? 1 : 0)) | (fused ? 0 : 0x100) | (fused_df ? 0 : 0x200))
    check(ctx, ccall((:mb200_csc_create, lib), Int32, (Ptr{Cvoid}, Ref{HParams}, Int64, Int32, Int32, Ref{Ptr{Cvoid}}),
                     ctx, hp, L, n_groups, flags, h))
    h[]
end
# flat = vcat(lambda_sparsity, kappa_sparsity, lambda_stepsize, omega_stepsize, kappa_stepsize, vec(D), vec(F), penalty_xyz, mu,
#             [lambda_sparsity_warmup, lambda_stepsize_warmup, omega_stepsize_warmup])   — Flux.params(cdl) order + warm-ups
csc_set_params(ctx, m, flat::Vector{Float32}) = GC.@preserve flat check(ctx, ccall((:mb200_csc_set_params, lib), Int32,
    (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}, Int64), ctx, m, flat, length(flat)))
function csc_get_params(ctx, m, n::Integer)
    flat = Vector{Float32}(undef, n)
    GC.@preserve flat check(ctx, ccall((:mb200_csc_get_params, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float32}, Int64), ctx, m, flat, n))
    flat
end
function train_step!(ctx, m, seqs, batch_idx0::Vector{Int64}; eta=1f-3, beta=(0.9f0, 0.999f0), eps=1f-8)
    GC.@preserve batch_idx0 check(ctx, ccall((:mb200_csc_step_begin, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}),
                                             ctx, m, seqs, batch_idx0))
    loss = Ref{Float32}(0); l1 = Ref{Float32}(0)
    check(ctx, ccall((:mb200_csc_adabelief_step, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Float32, Float32, Float32, Float32, Ref{Float32}, Ref{Float32}),
                     ctx, m, eta, beta[1], beta[2], eps, loss, l1))
    loss[], l1[]          # println("loss $(loss[])") keeps the reference's log (model.jl:392); stop when l1 < 95 (train.jl:47-52)
end

# replaces code_retrieval (inference/_1_code_retrieval.jl:33-56)
function code_retrieval(ctx, m, seqs, N::Integer, batch_size::Integer)
    n = N - N % batch_size
    cap = 64 * n; out = Vector{Code}(undef, cap); cnt = Ref{Int64}(0)
    GC.@preserve out check(ctx, ccall((:mb200_csc_codes, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ptr{Code}, Int64, Ref{Int64}),
                                      ctx, m, seqs, 0, n, out, cap, cnt))
    [(position=c.position + 0x0001, fil=c.fil + 0x0001, seq=c.seq + 0x00000001, mag=c.mag) for c in view(out, 1:cnt[])]
end

# replaces get_scanning_range_of_filtered_code_components + enumerate_triplets (inference/_2_enumerate.jl:25-65) and the key
# counting of get_enriched_keys (inference/_3_make_pfms.jl:3-26).  `codes` = the filtered stored_code_components (1-based fields).
struct KeyCount; key::UInt64; count::UInt32; reserved::UInt32; first::UInt64; end
struct TripletValue; key_index::UInt32; range_index::UInt32; position::UInt32; reserved::UInt32; order::UInt64; end
unpack_key(k::UInt64, h) = (f1=Int(k & 0xff), f2=Int((k >> 8) & 0xff), f3=Int((k >> 16) & 0xff), d12=Int((k >> 24) & 0xffff),
                            d13=Int((k >> 40) & 0xffff), len=Int((k >> 40) & 0xffff) + h)
function triplets_create(ctx, codes)
    pos = UInt16[c.position - 1 for c in codes]; fil = UInt16[c.fil - 1 for c in codes]; seq = UInt32[c.seq - 1 for c in codes]
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve pos fil seq check(ctx, ccall((:mb200_triplets_create, lib), Int32,
        (Ptr{Cvoid}, Ptr{UInt16}, Ptr{UInt16}, Ptr{UInt32}, Int64, Ref{Ptr{Cvoid}}, Ptr{Int64}, Ptr{Int64}), ctx, pos, fil, seq, length(pos), h, C_NULL, C_NULL))
    h[]
end
triplets_destroy(ctx, t) = ccall((:mb200_triplets_destroy, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ctx, t)
# keys with more than `min_count` values in Dictionary (first-insertion) order
function triplets_frequent(ctx, t, min_count::Integer)
    n = Ref{Int64}(0)
    check(ctx, ccall((:mb200_triplets_frequent, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{KeyCount}, Int64, Ref{Int64}), ctx, t, min_count, C_NULL, 0, n))
    out = Vector{KeyCount}(undef, n[])
    GC.@preserve out check(ctx, ccall((:mb200_triplets_frequent, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, UInt32, Ptr{KeyCount}, Int64, Ref{Int64}), ctx, t, min_count, out, n[], n))
    sort!(out, by = x -> x.first)
end
# get_enriched_keys(H; max_word_combinations, dec=-5, count_from=cover_more_than, count_to=cover_at_least) on the device dictionary
function get_enriched_keys(ctx, t; max_word_combinations=500, dec=-5, count_from=200, count_to=10, num_pfms2process=500)
    cand = triplets_frequent(ctx, t, count_to); enriched = KeyCount[]
    for count = count_from:dec:count_to
        enriched = filter(x -> x.count > count, cand)
        length(enriched) > max_word_combinations && return sort(enriched, by = x -> x.count, rev = true)[1:num_pfms2process]
    end
    enriched
end
# H[k] for the selected keys: Vector of [(seq_num = range index, pos)] in insertion order, as insert_H! builds them
function triplets_values(ctx, t, keys::Vector{KeyCount})
    ks = UInt64[k.key for k in keys]; total = sum(Int(k.count) for k in keys; init = 0)
    out = Vector{TripletValue}(undef, max(total, 1)); n = Ref{Int64}(0)
    GC.@preserve ks out check(ctx, ccall((:mb200_triplets_values, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{UInt64}, Int64, Ptr{TripletValue}, Int64, Ref{Int64}), ctx, t, ks, length(ks), out, total, n))
    recs = sort!(view(out, 1:n[]), by = v -> (v.key_index, v.order))
    H = [Tuple{Int,Int}[] for _ in keys]
    for v in recs push!(H[v.key_index + 1], (Int(v.range_index), Int(v.position))) end
    H
end

# Drop-in for pvalue2score (inference/_h2_Touzet.jl:170-187): returns `nothing` when no score qualifies.
function pvalue2score(pwm::AbstractMatrix, pval::Real, eps::Real=1e-1; bg=[.25, .25, .25, .25])
    rowmajor = collect(Float64, permutedims(pwm))            # C side reads 4 x m row-major = Julia (m,4) column-major
    bg64 = collect(Float64, bg); score = Ref{Float64}(0.0); found = Ref{Int32}(0)
    rc = GC.@preserve rowmajor bg64 ccall((:mb200_pvalue2score, lib), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int32, Float64, Float64, Ptr{Float64}, Ref{Float64}, Ref{Int32}),
        C_NULL, rowmajor, size(pwm, 2), pval, eps, bg64, score, found)
    rc == 0 || error("mb200_pvalue2score failed ($rc)")
    return found[] == 0 ? nothing : score[]
end

# Diagnostic: the int8 B operand of the tensor-core scan for one (motif, strand) slot. cols: (len, 4) Float16, row = PWM column in
# scoring order. Returns (e, k, Q) with Q (len, 4) Int8, or `nothing` when no window can exceed the threshold.
function scan_prefilter_int8(cols::AbstractMatrix{Float16}, thresh::Float16)
    len = size(cols, 1)
    rowmajor = collect(Float16, permutedims(cols))            # C side reads len x 4 row-major = Julia (4, len) column-major
    e = Ref{Int32}(0); possible = Ref{Int32}(0); k = zeros(Int32, len); q = zeros(Int8, 4, len)
    rc = GC.@preserve rowmajor k q ccall((:mb200_scan_prefilter_int8, lib), Int32,
        (Ptr{Float16}, Int32, UInt16, Ref{Int32}, Ptr{Int32}, Ptr{Int8}, Ref{Int32}),
        rowmajor, len, reinterpret(UInt16, thresh), e, k, q, possible)
    rc == 0 || error("mb200_scan_prefilter_int8 failed ($rc)")
    return possible[] == 0 ? nothing : (e[], k, permutedims(q))
end

# ------------------------------------------------------------------------------------------------------------------------------
# multi-GPU: one Julia process per GPU (Distributed / MPI / plain `julia -p`), one NCCL communicator per ctx (csrc/comm.cu).
# Rank 0 makes the id, the host ships the 128 bytes by its own means (e.g. `remotecall_fetch`), every rank calls comm_init.
# After that train_step! averages the gradients over ranks inside mb200_csc_adabelief_step, gpu_scan(...; reduce=true) and
# scan_hist(...; reduce=true) return sums over ranks, and code_retrieval(...; sharded=true) decodes 1/world of the batches per rank.
# ------------------------------------------------------------------------------------------------------------------------------
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    rc = GC.@preserve id ccall((:mb200_comm_unique_id, lib), Int32, (Ptr{UInt8},), id)
    rc == 0 || error("mb200_comm_unique_id failed ($rc): libnccl.so.2 not loadable")
    id
end
comm_init(ctx, id::Vector{UInt8}, rank::Integer, world::Integer) = GC.@preserve id check(ctx, ccall((:mb200_comm_init, lib), Int32,
    (Ptr{Cvoid}, Ptr{UInt8}, Int32, Int32), ctx, id, rank, world))
comm_destroy(ctx) = check(ctx, ccall((:mb200_comm_destroy, lib), Int32, (Ptr{Cvoid},), ctx))
function comm_info(ctx)
    r = Ref{Int32}(0); w = Ref{Int32}(1); v = Ref{Int32}(0)
    check(ctx, ccall((:mb200_comm_info, lib), Int32, (Ptr{Cvoid}, Ref{Int32}, Ref{Int32}, Ref{Int32}), ctx, r, w, v))
    (rank = Int(r[]), world = Int(w[]), nccl_version = Int(v[]))
end
# in-place broadcast of a bits-type array from `root` (epoch permutation seed, stop flag)
comm_broadcast!(ctx, a::Array, root::Integer=0) = (GC.@preserve a check(ctx, ccall((:mb200_comm_broadcast, lib), Int32,
    (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int32), ctx, a, sizeof(a), root)); a)
comm_allreduce!(ctx, a::Vector{Int64}) = (GC.@preserve a check(ctx, ccall((:mb200_comm_allreduce_i64, lib), Int32,
    (Ptr{Cvoid}, Ptr{Int64}, Int64), ctx, a, length(a))); a)
# start of data-parallel training: rank `root`'s weights and optimiser state become everybody's
csc_broadcast_params(ctx, m, root::Integer=0) = check(ctx, ccall((:mb200_csc_broadcast_params, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32), ctx, m, root))
# device addresses of the parameter / gradient vectors (for hosts that bring their own collective, e.g. NCCL.jl)
function csc_device_ptrs(m)
    p = Ref{Ptr{Cvoid}}(C_NULL); g = Ref{Ptr{Cvoid}}(C_NULL)
    ccall((:mb200_csc_device_ptrs, lib), Int32, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}, Ref{Ptr{Cvoid}}), m, p, g) == 0 || error("mb200_csc_device_ptrs")
    p[], g[]
end
# the per-step `S |> gpu` of train.jl:41 for hosts that keep the reads on the CPU: batch as L x 6 ASCII bytes (one column per read)
function train_step_host!(ctx, m, ascii_batch::Matrix{UInt8}; eta=1f-3, beta=(0.9f0, 0.999f0), eps=1f-8)
    GC.@preserve ascii_batch check(ctx, ccall((:mb200_csc_step_begin_host, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{UInt8}, Int64),
                                              ctx, m, ascii_batch, size(ascii_batch, 2)))
    loss = Ref{Float32}(0); l1 = Ref{Float32}(0)
    check(ctx, ccall((:mb200_csc_adabelief_step, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Float32, Float32, Float32, Float32, Ref{Float32}, Ref{Float32}),
                     ctx, m, eta, beta[1], beta[2], eps, loss, l1))
    loss[], l1[]
end
# code_retrieval sharded over the communicator's ranks (every rank gets all records, ordered by seq like the single-GPU call)
function code_retrieval_sharded(ctx, m, seqs, N::Integer, batch_size::Integer)
    n = N - N % batch_size
    cap = 64 * n; out = Vector{Code}(undef, cap); cnt = Ref{Int64}(0)
    GC.@preserve out check(ctx, ccall((:mb200_csc_codes_sharded, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Int32, Int32, Ptr{Code}, Int64, Ref{Int64}), ctx, m, seqs, 0, n, -1, -1, out, cap, cnt))
    [(position=c.position + 0x0001, fil=c.fil + 0x0001, seq=c.seq + 0x00000001, mag=c.mag) for c in view(out, 1:cnt[])]
end

# ------------------------------------------------------------------------------------------------------------------------------
# seam S4 (SURVEY §8b): thresholds, filter, counts, Fisher without hit dictionaries
# ------------------------------------------------------------------------------------------------------------------------------
# (32768, K) histogram of the Float16 bit patterns of all hit scores (score > 0, both strands): the input of get_max_score /
# get_min_score / the sweep of get_best_thresh (inference/_s2_filter_pos_w_scores.jl:11-36, 99-113)
function scan_hist(ctx, seqs, pwms::Array{Float16,3}, lens::Vector{Int64}; reduce=false)
    K, _, maxlen = size(pwms)
    hist = zeros(UInt32, 32768, K)
    GC.@preserve pwms lens hist check(ctx, ccall((:mb200_scan_hist, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float16}, Ptr{Int64}, Int32, Int32, UInt32, Ptr{UInt32}),
        ctx, seqs, pwms, lens, K, maxlen, SCAN_FWD | SCAN_RC | (reduce ? SCAN_REDUCE : UInt32(0)), hist))
    hist
end
# best site per (sequence, motif) over every window greedy_search! scores (_h3_1_alignment.jl:18-36), both strands by default:
# (K, N) NamedTuples with 1-based `pos` (0 when not found), `comp` (true = reverse(pwm)), `score`, `found`.  Ties: smaller
# position, then the forward strand.  The per-sequence feature behind AUC / central-enrichment statistics.
function scan_best(ctx, seqs, N::Integer, pwms::Array{Float16,3}, lens::Vector{Int64}; fwd=true, rc=true)
    K, _, maxlen = size(pwms)
    out = Matrix{Best}(undef, K, N)                                    # row-major (N, K) in C = (K, N) in Julia
    GC.@preserve pwms lens out check(ctx, ccall((:mb200_scan_best, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float16}, Ptr{Int64}, Int32, Int32, UInt32, Ptr{Best}),
        ctx, seqs, pwms, lens, K, maxlen, (fwd ? SCAN_FWD : UInt32(0)) | (rc ? SCAN_RC : UInt32(0)), out))
    [(pos = b.found != 0 ? Int(b.pos) + 1 : 0, comp = b.comp != 0, score = b.score, found = b.found != 0) for b in out]
end

# windows [start, start + len) of rows `row` (1-based rows and starts) as a new fixed-length store (mb200_seqs_windows)
function seqs_windows(ctx, seqs, row::Vector{Int64}, start::Vector{Int64}, len::Integer)
    length(row) == length(start) || error("row and start must have one length")
    r0, s0 = row .- 1, start .- 1
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve r0 s0 check(ctx, ccall((:mb200_seqs_windows, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Int64, Int64, Ref{Ptr{Cvoid}}), ctx, seqs, r0, s0, length(r0), len, out))
    out[]
end

struct Anchor                      # mb200_anchor (24 bytes), 0-based inside
    row::Int64
    start::Int64
    len::Int32
    primary::UInt16
    comp::UInt8
    _pad::UInt8
end

# SpaMo spacing histogram (mb200_scan_spacing).  Anchors: (row, start, len, primary, comp) with 1-based row, start and primary;
# returns hist as an Int array (margin, 4, K, n_primary) in Julia order = hist[g+1, q+1, k, p] with gap g and quadrant q (0 same
# strand upstream, 1 same downstream, 2 opposite upstream, 3 opposite downstream), and with want_sites the (K, n) best sites of
# every (anchor, secondary) as NamedTuples (1-based pos in the row, found = counted).
function scan_spacing(ctx, seqs, anchors::Vector{<:NamedTuple}, n_primary::Integer, pwms::Array{Float16,3}, lens::Vector{Int64};
                      margin::Integer=150, thresh::Union{Nothing,Vector{Float16}}=nothing, want_sites::Bool=false)
    K, _, maxlen = size(pwms)
    an = [Anchor(a.row - 1, a.start - 1, Int32(a.len), UInt16(a.primary - 1), UInt8(a.comp), 0x00) for a in anchors]
    hist = zeros(UInt32, margin, 4, K, n_primary)
    sites = want_sites ? Matrix{Best}(undef, K, length(an)) : Matrix{Best}(undef, 0, 0)
    tp = thresh === nothing ? Ptr{Float16}(C_NULL) : pointer(thresh)
    sp = want_sites ? pointer(sites) : Ptr{Best}(C_NULL)
    GC.@preserve an pwms lens thresh hist sites check(ctx, ccall((:mb200_scan_spacing, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Anchor}, Int64, Int32, Int32, Ptr{Float16}, Ptr{Int64}, Int32, Int32, Ptr{Float16}, Ptr{UInt32}, Ptr{Best}),
        ctx, seqs, an, length(an), n_primary, margin, pwms, lens, K, maxlen, tp, hist, sp))
    st = want_sites ? [(pos = b.pos == typemax(UInt32) ? 0 : Int(b.pos) + 1, comp = b.comp != 0, score = b.score, found = b.found != 0) for b in sites] : nothing
    Int.(hist), st
end

# fused scan + filter_position_by_best_thresh! + get_uniq_counts + union_ranges coverage: (4, K) Int64, rows = hits, unique starts,
# coverage as the reference computes it (_h4_overlap_ratio.jl:48-56), true coverage
scan_counts(ctx, seqs, pwms, lens, thresh::Vector{Float16}; reduce=false) =
    gpu_scan(ctx, seqs, pwms, lens; thresh=thresh, want_hits=false, reduce=reduce)[4]

# get_best_thresh (_s2:90-114) from the two histograms.  `fisher(a, b)` is the host's right-tail test, e.g.
#   (a, b) -> pvalue(FisherExactTest(a, asum - a, b, asum - b), tail=:right)        (HypothesisTests, as in the reference)
function best_thresh_from_hist(h_fg::AbstractVector{UInt32}, h_bg::AbstractVector{UInt32}, eff_pos, pwm, bg, fisher;
                               touzet_len=15, increment=Float16(0.5), pvalue_of=n -> (n <= 11 ? (n <= 9 ? 3e-4 : 1e-4) : 1e-4))
    if any(length(r) < touzet_len for r in eff_pos)
        best = 0.0
        for r in eff_pos
            (length(r) > touzet_len || length(r) <= 1) && continue
            sub = view(pwm, :, r)
            best += pvalue2score(sub, pvalue_of(size(sub, 2)); bg=bg)
        end
        return Float16(best)
    end
    nz = findall(i -> h_fg[i] + h_bg[i] > 0, 1:0x7C01)                 # positive finite halves and +Inf, ascending in value
    isempty(nz) && return Float16(Inf)
    min_score = reinterpret(Float16, UInt16(nz[1] - 1)); max_score = reinterpret(Float16, UInt16(nz[end] - 1))
    tail_fg = reverse(cumsum(reverse(Int64.(h_fg)))); tail_bg = reverse(cumsum(reverse(Int64.(h_bg))))    # tail[b+1] = hits with pattern >= b
    best_thresh, t, best_p = min_score, min_score, 1.0
    while t < max_score
        b = Int(reinterpret(UInt16, t))
        a_, b_ = b + 2 <= 32768 ? tail_fg[b + 2] : 0, b + 2 <= 32768 ? tail_bg[b + 2] : 0      # scores strictly greater than t
        p = fisher(a_, b_)
        if p < best_p; best_p = p; best_thresh = t; end
        t = Float16(t + increment)
    end
    best_thresh
end

# body of filter_positions_scores_usecomp!(ms, data, bg) (_s2_filter_pos_w_scores.jl:127-138) on the library: two histogram scans
# give ms.score_thresh, two fused counting scans give the filtered occurrence counts (fg, bg) — no positions/scores dictionaries.
function filter_positions_scores_usecomp!(ctx, ms, seqs_fg, seqs_bg, pwms, NL::Integer, bg, fisher)
    h_fg = scan_hist(ctx, seqs_fg, pwms, ms.lens); h_bg = scan_hist(ctx, seqs_bg, pwms, ms.lens)
    ms.score_thresh = [best_thresh_from_hist(view(h_fg, :, k), view(h_bg, :, k), ms.effective_segments[k], ms.pwms[k], bg,
                                             (a, b) -> fisher(a, NL - a, b, NL - b)) for k in 1:length(ms.lens)]
    scan_counts(ctx, seqs_fg, pwms, ms.lens, ms.score_thresh), scan_counts(ctx, seqs_bg, pwms, ms.lens, ms.score_thresh)
end

# body of pvec_from_test_data(ms, data) (render/pvec_calculations.jl:1-22): test-set scans filtered by ms.score_thresh, union
# coverage (row 3), Fisher; returns (pvec, uniq_active_counts_test)
function pvec_from_test_data(ctx, ms, seqs_test, seqs_bg_test, pwms, NL_test::Integer, fisher)
    c = scan_counts(ctx, seqs_test, pwms, ms.lens, ms.score_thresh); cb = scan_counts(ctx, seqs_bg_test, pwms, ms.lens, ms.score_thresh)
    pvec = [(c[3, k] == 0 && cb[3, k] == 0) ? 1.0 : fisher(c[3, k], NL_test - c[3, k], cb[3, k], NL_test - cb[3, k]) for k in 1:length(ms.lens)]
    pvec, Float64.(c[2, :])
end

# exact p-values of greedy_search!'s Float16 score (new): survival tables of every (motif, strand) under an independent-base
# background bg (A, C, G, T), built on the device; the handle owns them until pvtab_destroy.  pwms / lens as for gpu_scan.
function pvtab_create(ctx, pwms::Array{Float16,3}, lens::Vector{Int64}, bg::Vector{Float64})
    K, _, maxlen = size(pwms)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve pwms lens bg check(ctx, ccall((:mb200_pvtab_create, lib), Int32,
        (Ptr{Cvoid}, Ptr{Float16}, Ptr{Int64}, Int32, Int32, Ptr{Float64}, Ref{Ptr{Cvoid}}), ctx, pwms, lens, K, maxlen, bg, h))
    h[]
end
pvtab_destroy(ctx, t) = ccall((:mb200_pvtab_destroy, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ctx, t)
# (2, K) Float16 thresholds, column k = (forward, reverse(pwm)): score > thresh <=> p-value <= pval[k]
function pvtab_thresholds(ctx, t, pval::Vector{Float64})
    out = zeros(Float16, 2, length(pval))
    GC.@preserve pval out check(ctx, ccall((:mb200_pvtab_thresholds, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float16}), ctx, t, pval, out))
    out
end
# p-values of hits (1-based motif, comp = true for reverse(pwm)); NaN for a NaN score
function pvtab_lookup(ctx, t, motif::Vector{<:Integer}, comp::AbstractVector{Bool}, score::Vector{Float16})
    m0, c0 = UInt16.(motif .- 1), UInt8.(comp)
    p = zeros(Float64, length(score))
    GC.@preserve m0 c0 score p check(ctx, ccall((:mb200_pvtab_lookup, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{UInt16}, Ptr{UInt8}, Ptr{Float16}, Int64, Ptr{Float64}), ctx, t, m0, c0, score, length(score), p))
    p
end
# the whole table of (motif k, strand comp): 65536 Float64 indexed by Float16 bit pattern + 1, NaN for the NaN patterns
function pvtab_survival(ctx, t, k::Integer, comp::Bool)
    out = zeros(Float64, 65536)
    GC.@preserve out check(ctx, ccall((:mb200_pvtab_survival, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Ptr{Float64}), ctx, t, k - 1, Int32(comp), out))
    out
end

# positions -> count matrices: posdicts2countmats / msa_add! (inference/_h6_positions2countmat.jl:7-54).  sites: 0-based
# (motif, seq, pos, comp) rows; returns Vector of 4 x len_k UInt32 matrices (add the 0.01 pseudo-count and convert on the host).
struct Site; motif::UInt32; seq::UInt32; pos::UInt32; comp::UInt32; end
function count_matrices(ctx, seqs, sites::Vector{Site}, lens::Vector{Int64})
    K = length(lens); maxlen = Int(maximum(lens))
    counts = zeros(UInt32, 4, maxlen, K)                               # C side: [(k*maxlen + col)*4 + base]
    GC.@preserve sites lens counts check(ctx, ccall((:mb200_count_matrices, lib), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Site}, Int64, Ptr{Int64}, Int32, Int32, Ptr{UInt32}), ctx, seqs, sites, length(sites), lens, K, maxlen, counts))
    [counts[:, 1:lens[k], k] for k in 1:K]
end

end # module
