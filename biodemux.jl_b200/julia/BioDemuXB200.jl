# BioDemuXB200.jl -- ccall shim that swaps BioDemuX.jl's CPU worker loop for libbdx.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: Julia is not installed in the build image, so
# this file is delivered as the reference-side binding a BioDemuX maintainer would add
# (see INTEGRATION.md).  The same call sequence is exercised from Python (ctypes) in
# biodemux.jl_b200/capi.py and tests/test_gpu_parity.py.
#
# It replaces the body of `worker_task` (BioDemuX src/core.jl:226-279): for every Chunk it
# packs the read-1 sequences, lets the GPU classify them and rebuilds exactly what the
# CPU loop produced -- `filenames::Vector{String}` and `trim_ranges` -- so reader_task,
# writer_task and generate_summary_report stay untouched.
module BioDemuXB200

using BioDemuX
using BioDemuX: DemuxConfig, DemuxStats, DynamicRange, Chunk, ResultChunk

const libbdx = get(ENV, "LIBBDX", joinpath(@__DIR__, "..", "csrc", "libbdx.so"))
const BDX_ABI_VERSION = UInt32(1)

# ---- struct mirrors of include/bdx.h (field order and widths must match) -----------------
struct BdxRange            # bdx_range  <- DynamicRange (classification.jl:9-14)
    start_offset::Int64
    start_from_end::Int32
    end_from_end::Int32
    end_offset::Int64
end
BdxRange(r::DynamicRange) = BdxRange(r.start_offset, r.start_from_end, r.end_from_end, r.end_offset)

struct BdxBarcodeSet       # bdx_barcode_set
    n_barcodes::Int32
    trim_side::Int32
    bytes::Ptr{UInt8}
    offsets::Ptr{Int32}
    lengths_no_n::Ptr{Int32}
    ref_search_range::BdxRange
    barcode_start_range::BdxRange
    barcode_end_range::BdxRange
end

struct BdxParams           # bdx_params <- DemuxConfig (classification.jl:16-58)
    struct_size::UInt32
    abi_version::UInt32
    max_error_rate::Float64
    min_delta::Float64
    match::Int64
    mismatch::Int64
    indel::Int64
    nindel::Int64
    has_nindel::Int32
    algorithm::Int32
    is_dual::Int32
    want_stats::Int32
    set1::BdxBarcodeSet
    set2::BdxBarcodeSet
end

struct BdxResult           # bdx_result
    status::Int32
    bc1::Int32
    bc2::Int32
    keep_start::Int32
    keep_end::Int32
end

struct BdxStatsOverflow    # bdx_stats_overflow
    pass::Int32
    bc::Int32
    start::Int32
    length::Int32
end

struct BdxStatsLayout      # bdx_stats_layout
    total_len::Int64
    sample_off::Int64
    b1::Int32
    b2::Int32
    pos_bins::Int32
    len_bins::Int32
    dist_bins::Int32
    pos_bias::Int32
    dist_bias::Int32
    reserved::Int32
    pos_off::NTuple{2,Int64}
    len_off::NTuple{2,Int64}
    dist_off::NTuple{2,Int64}
end

bdx_error() = unsafe_string(ccall((:bdx_last_error, libbdx), Cstring, ()))
check(rc) = rc == 0 ? nothing : error("libbdx: $(bdx_error()) (code $rc)")

algorithm_code(s::Symbol) = s == :hamming ? Int32(1) : s == :exact ? Int32(2) : Int32(0)  # classification.jl:639-649

# Keeps the Julia arrays the C structs point into alive.
mutable struct GpuConfig
    handle::Ptr{Cvoid}
    config::DemuxConfig
    keep::Vector{Any}
end

function pack_set(keep, seqs::Vector{String}, lens::Vector{Int}, rs, bs, be, trim)
    bytes = Vector{UInt8}(join(seqs))
    offsets = Int32[0; cumsum(ncodeunits.(seqs))]
    lens32 = isempty(lens) ? Int32[0] : Int32.(lens)
    push!(keep, bytes, offsets, lens32)
    BdxBarcodeSet(length(seqs), isnothing(trim) ? 0 : trim, pointer(bytes), pointer(offsets), pointer(lens32),
                  BdxRange(rs), BdxRange(bs), BdxRange(be))
end

function GpuConfig(c::DemuxConfig)
    keep = Any[]
    set1 = pack_set(keep, c.bc_seqs, c.bc_lengths_no_N, c.ref_search_range, c.barcode_start_range,
                    c.barcode_end_range, c.trim_side)
    set2 = c.is_dual ?
        pack_set(keep, c.bc_seqs2, c.bc_lengths_no_N2, c.ref_search_range2, c.barcode_start_range2,
                 c.barcode_end_range2, c.trim_side2) : set1
    p = Ref(BdxParams(sizeof(BdxParams), BDX_ABI_VERSION, c.max_error_rate, c.min_delta, c.match, c.mismatch,
                      c.indel, something(c.nindel, 0), isnothing(c.nindel) ? 0 : 1,
                      algorithm_code(c.matching_algorithm), c.is_dual ? 1 : 0, c.summary ? 1 : 0, set1, set2))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve keep check(ccall((:bdx_config_create, libbdx), Cint, (Ref{BdxParams}, Ref{Ptr{Cvoid}}), p, h))
    g = GpuConfig(h[], c, keep)
    finalizer(x -> ccall((:bdx_config_destroy, libbdx), Cvoid, (Ptr{Cvoid},), x.handle), g)
    g
end

# classification.jl:877-900 -- filename is a pure function of (status, bc1, bc2)
function filename_of(c::DemuxConfig, r::BdxResult)
    suffix = c.gzip_output ? ".fastq.gz" : ".fastq"
    r.status == 1 && return "unknown" * suffix
    r.status == 2 && return "ambiguous_classification" * suffix
    c.is_dual ? string(c.ids[r.bc1]) * "." * string(c.ids2[r.bc2]) * suffix : string(c.ids[r.bc1]) * suffix
end

"""
    gpu_worker_task(input_channel, output_channel, gcfg; device=0, chunk_size=4000, max_read_len=1024, windows=false)

Drop-in for `BioDemuX.worker_task` (core.jl:226-279).  One bdx_stream per worker task; up to three batches are
kept in flight so H2D copies overlap the kernels.  The stream's pinned staging holds `chunk_size` reads /
`chunk_size * max_read_len` sequence bytes per batch: a chunk that does not fit (long reads, or a reader chunk
larger than the worker's) is split into several batches -- nothing is ever written past the staging buffers --
and only a single read longer than the whole staging buffer is an error (raise `max_read_len`).  With
`windows=true` only the bytes of every read's search windows travel (`bdx_submit_windows`; same results): the gain
of long reads with short search ranges.  Returns the stream's DemuxStats (from the device counters) when
`config.summary`, else `nothing`.
"""
function gpu_worker_task(input_channel::Channel{Chunk}, output_channel::Channel{ResultChunk}, g::GpuConfig;
                         device::Int=0, chunk_size::Int=4000, max_read_len::Int=1024, windows::Bool=false)
    c = g.config
    max_bytes = chunk_size * max_read_len
    sref = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:bdx_stream_create, libbdx), Cint, (Ptr{Cvoid}, Cint, Int32, Int64, Ref{Ptr{Cvoid}}),
                g.handle, device, chunk_size, max_bytes, sref))
    s = sref[]
    do_trim = !isnothing(c.trim_side) || !isnothing(c.trim_side2)
    # a chunk and the result arrays its batches fill; `left` = batches of it not yet fetched
    pending = Tuple{Chunk,Vector{String},Union{Vector{Union{UnitRange{Int},Nothing}},Nothing},Base.RefValue{Int}}[]
    in_flight = Tuple{Int,UnitRange{Int}}[]          # (index into pending, reads of that chunk), oldest first
    results = Vector{BdxResult}(undef, chunk_size)

    function finish_oldest()
        (_, rng) = popfirst!(in_flight)
        chunk, filenames, trim_ranges, left = pending[1]
        tag = Ref{UInt64}(0); nn = Ref{Int32}(0)
        check(ccall((:bdx_fetch, libbdx), Cint, (Ptr{Cvoid}, Ref{UInt64}, Ref{Int32}, Ptr{BdxResult}, Ptr{Cvoid}),
                    s, tag, nn, results, C_NULL))
        nn[] == length(rng) || error("libbdx: batch of $(length(rng)) reads came back with $(nn[]) results")
        @inbounds for (k, i) in enumerate(rng)
            r = results[k]
            filenames[i] = filename_of(c, r)
            if do_trim                                   # core.jl:249-255
                trim_ranges[i] = r.keep_start != -1 ? (Int(r.keep_start):Int(r.keep_end)) : nothing
            end
        end
        left[] -= 1
        if left[] == 0                                   # batches come back in submission order: chunks stay ordered
            popfirst!(pending)
            put!(output_channel, ResultChunk(chunk, filenames, trim_ranges))
        end
    end

    try
        for chunk in input_channel
            seqs = chunk.data.seqs
            n = length(seqs)
            # split the chunk into batches that fit the staging buffers (usually exactly one)
            ranges = UnitRange{Int}[]
            first_i, bytes = 1, 0
            for i in 1:n
                len = ncodeunits(seqs[i])
                len > max_bytes && error("libbdx: a read of $len bases exceeds the worker's staging buffer " *
                                         "($max_bytes bytes); create it with a larger max_read_len")
                if i - first_i >= chunk_size || bytes + len > max_bytes
                    push!(ranges, first_i:i-1)
                    first_i, bytes = i, 0
                end
                bytes += len
            end
            push!(ranges, first_i:n)
            push!(pending, (chunk, Vector{String}(undef, n),
                            do_trim ? Vector{Union{UnitRange{Int},Nothing}}(undef, n) : nothing, Ref(length(ranges))))
            for rng in ranges
                while length(in_flight) >= 3                 # BDX_MAX_IN_FLIGHT is 4
                    finish_oldest()
                end
                if windows
                    submit_windows(s, g, seqs, rng, chunk.id)
                    push!(in_flight, (length(pending), rng))
                    continue
                end
                # zero-copy: write straight into the stream's pinned staging (bounds established above)
                pseq = Ref{Ptr{UInt8}}(C_NULL); poff = Ref{Ptr{Int32}}(C_NULL)
                check(ccall((:bdx_acquire, libbdx), Cint, (Ptr{Cvoid}, Ref{Ptr{UInt8}}, Ref{Ptr{Int32}}), s, pseq, poff))
                off = 0
                unsafe_store!(poff[], Int32(0), 1)
                @inbounds for (k, i) in enumerate(rng)
                    len = ncodeunits(seqs[i])
                    @assert off + len <= max_bytes && k <= chunk_size
                    GC.@preserve seqs unsafe_copyto!(pseq[] + off, pointer(seqs[i]), len)
                    off += len
                    unsafe_store!(poff[], Int32(off), k + 1)
                end
                check(ccall((:bdx_commit, libbdx), Cint, (Ptr{Cvoid}, Int32, UInt64), s, length(rng), chunk.id))
                push!(in_flight, (length(pending), rng))
            end
            while length(in_flight) > 2
                finish_oldest()
            end
        end
        while !isempty(in_flight)
            finish_oldest()
        end
        return c.summary ? fetch_stats(s, g) : nothing
    finally
        ccall((:bdx_stream_destroy, libbdx), Cvoid, (Ptr{Cvoid},), s)
    end
end

"bdx_window_spans: ([lo1, hi1, lo2, hi2], window length) of a read of `len` bases (1-based, inclusive; hi < lo = empty)."
function window_spans(g::GpuConfig, len::Integer)
    sp = zeros(Int32, 4)
    n = ccall((:bdx_window_spans, libbdx), Cint, (Ptr{Cvoid}, Int32, Ptr{Int32}), g.handle, len, sp)
    n < 0 && error("libbdx: " * bdx_error())
    return sp, Int(n)
end

"One batch as the reads' window bytes (bdx_submit_windows; the library copies them to its staging before returning)."
function submit_windows(s::Ptr{Cvoid}, g::GpuConfig, seqs::Vector{String}, rng::UnitRange{Int}, tag)
    off = zeros(Int32, length(rng) + 1)
    woff = zeros(Int32, length(rng) + 1)
    win = UInt8[]
    spans = Dict{Int,Tuple{Vector{Int32},Int}}()      # the spans follow from the length alone
    for (k, i) in enumerate(rng)
        cu = codeunits(seqs[i])
        sp, wl = get!(() -> window_spans(g, length(cu)), spans, length(cu))
        for j in (1, 3)
            sp[j+1] >= sp[j] && append!(win, view(cu, sp[j]:sp[j+1]))
        end
        off[k+1] = off[k] + length(cu)
        woff[k+1] = woff[k] + wl
    end
    check(ccall((:bdx_submit_windows, libbdx), Cint,
                (Ptr{Cvoid}, Ptr{UInt8}, Ptr{Int32}, Ptr{Int32}, Int32, Cint, UInt64),
                s, win, woff, off, length(rng), 0, tag))
end

"Device counters -> DemuxStats (classification.jl:736-767); score keys are round(dist / norm, digits=2)."
function fetch_stats(s::Ptr{Cvoid}, g::GpuConfig)
    c = g.config
    lay = Ref{BdxStatsLayout}()
    check(ccall((:bdx_stats_layout_get, libbdx), Cint, (Ptr{Cvoid}, Ref{BdxStatsLayout}), g.handle, lay))
    L = lay[]
    buf = Vector{Int64}(undef, L.total_len)
    check(ccall((:bdx_stats_fetch, libbdx), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64), s, buf, length(buf)))
    st = DemuxStats()
    st.total_reads, st.matched_reads, st.unmatched_reads, st.ambiguous_reads = buf[1], buf[2], buf[3], buf[4]
    for b1 in 0:L.b1, b2 in 0:L.b2
        v = buf[L.sample_off + b1 * (L.b2 + 1) + b2 + 1]
        v > 0 && (st.sample_counts[(b1, b2)] = v)
    end
    norm_of(pass, b) = begin
        seqs = pass == 1 ? c.bc_seqs : c.bc_seqs2
        lens = pass == 1 ? c.bc_lengths_no_N : c.bc_lengths_no_N2
        (c.matching_algorithm != :hamming && c.matching_algorithm != :exact && !isnothing(c.nindel)) ?
            lens[b] : ncodeunits(seqs[b])
    end
    for pass in 1:(c.is_dual ? 2 : 1)
        nb = pass == 1 ? L.b1 : L.b2
        gpos, glen, gsc, pbs, pbp, pbl = pass == 1 ?
            (st.bc1_pos_counts, st.bc1_len_counts, st.bc1_score_counts, st.bc1_per_bc_score_counts,
             st.bc1_per_bc_pos_counts, st.bc1_per_bc_len_counts) :
            (st.bc2_pos_counts, st.bc2_len_counts, st.bc2_score_counts, st.bc2_per_bc_score_counts,
             st.bc2_per_bc_pos_counts, st.bc2_per_bc_len_counts)
        for b in 0:nb
            for k in 0:L.pos_bins-1
                v = buf[L.pos_off[pass] + b * L.pos_bins + k + 1]; v == 0 && continue
                b == 0 ? (gpos[k - L.pos_bias] = v) : (get!(() -> Dict{Int,Int}(), pbp, b)[k - L.pos_bias] = v)
            end
            for k in 0:L.len_bins-1
                v = buf[L.len_off[pass] + b * L.len_bins + k + 1]; v == 0 && continue
                b == 0 ? (glen[k] = v) : (get!(() -> Dict{Int,Int}(), pbl, b)[k] = v)
            end
            b == 0 && continue
            for d in 0:L.dist_bins-1
                v = buf[L.dist_off[pass] + b * L.dist_bins + d + 1]; v == 0 && continue
                key = round((d - L.dist_bias) / norm_of(pass, b), digits=2)
                dd = get!(() -> Dict{Float64,Int}(), pbs, b)
                dd[key] = get(dd, key, 0) + v
                gsc[key] = get(gsc, key, 0) + v
            end
        end
    end
    # matched passes whose start / length lies outside the device histograms (long reads searched near
    # their end) come back as exact records
    n, lost = Ref{Int64}(0), Ref{Int64}(0)
    check(ccall((:bdx_stats_overflow_fetch, libbdx), Cint, (Ptr{Cvoid}, Ptr{BdxStatsOverflow}, Int64, Ref{Int64}, Ref{Int64}),
                s, C_NULL, 0, n, lost))
    lost[] == 0 || error("libbdx: $(lost[]) stats overflow records were lost")
    ovf = Vector{BdxStatsOverflow}(undef, n[])
    n[] > 0 && check(ccall((:bdx_stats_overflow_fetch, libbdx), Cint,
                           (Ptr{Cvoid}, Ptr{BdxStatsOverflow}, Int64, Ref{Int64}, Ref{Int64}), s, ovf, length(ovf), n, lost))
    for e in ovf
        gpos, glen, pbp, pbl = e.pass == 1 ?
            (st.bc1_pos_counts, st.bc1_len_counts, st.bc1_per_bc_pos_counts, st.bc1_per_bc_len_counts) :
            (st.bc2_pos_counts, st.bc2_len_counts, st.bc2_per_bc_pos_counts, st.bc2_per_bc_len_counts)
        gpos[e.start] = get(gpos, e.start, 0) + 1
        glen[e.length] = get(glen, e.length, 0) + 1
        dp = get!(() -> Dict{Int,Int}(), pbp, Int(e.bc)); dp[e.start] = get(dp, e.start, 0) + 1
        dl = get!(() -> Dict{Int,Int}(), pbl, Int(e.bc)); dl[e.length] = get(dl, e.length, 0) + 1
    end
    st
end

# ---- device FASTQ path (bdx_demux_block): replaces reader_task's record splitting and writer_task's
# per-record trimming / routing (core.jl:43-224).  The Julia host keeps file I/O and (de)compression.
struct BdxDemuxBucket      # bdx_demux_bucket
    status::Int32
    bc1::Int32
    bc2::Int32
    n_records::Int32
    offset1::Int64
    length1::Int64
    offset2::Int64
    length2::Int64
end

struct BdxDemuxOut         # bdx_demux_out
    n_records::Int32
    n_buckets::Int32
    consumed1::Int64
    consumed2::Int64
    out1::Ptr{UInt8}
    out1_len::Int64
    out2::Ptr{UInt8}
    out2_len::Int64
    buckets::Ptr{BdxDemuxBucket}
    results::Ptr{BdxResult}
end

const BDX_DEMUX_SINGLE, BDX_DEMUX_MATES, BDX_DEMUX_BOTH = Cint(0), Cint(1), Cint(2)

"""
    demux_block!(handles, s, c, block1, block2, final, mode, prefix1, prefix2)

One block of FASTQ text per input through `bdx_demux_block`; every returned bucket is appended to its
output file (`handles(filename)::IO` is writer_task's `get_handle`, core.jl:122-132).  Returns
`(n_records, consumed1, consumed2)`; the caller re-presents `block[consumed+1:end]` in front of the next block
and stops once a final block has been consumed completely (`while !eof(io1) && !eof(io2)`, core.jl:48).
"""
function demux_block!(handles, s::Ptr{Cvoid}, c::DemuxConfig, block1::Vector{UInt8}, block2::Union{Vector{UInt8},Nothing},
                      final::Integer, mode::Cint, prefix1::String, prefix2::String)
    out = Ref{BdxDemuxOut}()
    b2 = isnothing(block2) ? UInt8[] : block2
    GC.@preserve block1 b2 check(ccall((:bdx_demux_block, libbdx), Cint,
        (Ptr{Cvoid}, Ptr{UInt8}, Int64, Ptr{UInt8}, Int64, Cint, Cint, Ref{BdxDemuxOut}),
        s, block1, length(block1), b2, length(b2), final, mode, out))
    o = out[]
    for k in 1:o.n_buckets
        b = unsafe_load(o.buckets, k)
        name = filename_of(c, BdxResult(b.status, b.bc1, b.bc2, -1, -1))
        if mode != BDX_DEMUX_MATES
            unsafe_write(handles(prefix1 * "." * name), o.out1 + b.offset1, b.length1)
        end
        if mode != BDX_DEMUX_SINGLE
            unsafe_write(handles(prefix2 * "." * name), o.out2 + b.offset2, b.length2)
        end
    end
    (o.n_records, o.consumed1, o.consumed2)
end

# ---- barcode tables through the C++ loader (preprocess_bc_file twin, fileio.jl:7-72) ------------------
function load_barcode_table(path::String, complement::Bool, rev::Bool)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:bdx_barcode_table_load, libbdx), Cint, (Cstring, Cint, Cint, Ref{Ptr{Cvoid}}), path, complement, rev, h)
    rc == 0 || error(unsafe_string(ccall((:bdx_barcode_table_error, libbdx), Cstring, ())))
    t = h[]
    n = ccall((:bdx_barcode_table_count, libbdx), Int32, (Ptr{Cvoid},), t)
    nid = ccall((:bdx_barcode_table_id_count, libbdx), Int32, (Ptr{Cvoid},), t)
    off = unsafe_wrap(Array, ccall((:bdx_barcode_table_offsets, libbdx), Ptr{Int32}, (Ptr{Cvoid},), t), n + 1)
    bytes = ccall((:bdx_barcode_table_bytes, libbdx), Ptr{UInt8}, (Ptr{Cvoid},), t)
    lens = n == 0 ? Int[] : Int.(unsafe_wrap(Array, ccall((:bdx_barcode_table_lengths_no_n, libbdx), Ptr{Int32}, (Ptr{Cvoid},), t), n))
    seqs = [unsafe_string(bytes + off[i], off[i+1] - off[i]) for i in 1:n]
    ids = [unsafe_string(ccall((:bdx_barcode_table_id, libbdx), Cstring, (Ptr{Cvoid}, Int32), t, i - 1)) for i in 1:nid]
    ccall((:bdx_barcode_table_destroy, libbdx), Cvoid, (Ptr{Cvoid},), t)
    seqs, lens, ids
end

end # module
