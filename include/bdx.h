/*
 * bdx.h -- C ABI of libbdx, the B200-native barcode-assignment engine.
 *
 * Drop-in boundary: the body of BioDemuX.jl's `worker_task`
 * (reference src/core.jl:226-279): given a chunk of read-1 sequences and an
 * immutable DemuxConfig, produce per read (status, barcode index/indices,
 * keep range) and -- when a summary is requested -- the per-worker DemuxStats
 * counters.  The reference has no FFI of its own; INTEGRATION.md shows the
 * `ccall` shim a BioDemuX maintainer adds to replace that loop body.
 *
 * Conventions
 *  - plain C types only; every call returns BDX_OK (0) or a negative bdx_status
 *    and never throws, aborts or exits;  bdx_last_error() gives the message of
 *    the last failure on the calling thread;
 *  - there is NO CPU fallback: if no sm_100 device/driver is usable the calls
 *    that need one return BDX_ERR_CUDA;
 *  - positions are 1-based inclusive, barcode indices are 1-based (0 = none),
 *    exactly as in the reference;
 *  - a bdx_config is immutable and may be shared by any number of streams and
 *    threads; a bdx_stream is owned by one thread at a time (it mirrors the
 *    per-worker SemiGlobalWorkspace, core.jl:229-233).
 */
#ifndef BDX_H
#define BDX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BDX_ABI_VERSION 1
#define BDX_MAX_IN_FLIGHT 4 /* batches a stream keeps in flight (ring of staging slots) */

typedef enum bdx_status {
    BDX_OK = 0,
    BDX_ERR_INVALID = -1,     /* bad argument / unsupported option value */
    BDX_ERR_CUDA = -2,        /* CUDA runtime error or no usable device */
    BDX_ERR_NOMEM = -3,
    BDX_ERR_STATE = -4,       /* call sequence error (fetch with nothing in flight, ...) */
    BDX_ERR_TOO_LARGE = -5    /* batch exceeds the stream's max_reads / max_bytes */
} bdx_status;

/* matching_algorithm (classification.jl:57, :639-649) */
typedef enum bdx_algorithm {
    BDX_SEMIGLOBAL = 0, /* semiglobal_alignment[_N]   classification.jl:238-477 */
    BDX_HAMMING = 1,    /* hamming_align              classification.jl:557-625 */
    BDX_EXACT = 2       /* exact_align                classification.jl:485-548 */
} bdx_algorithm;

/* per-read status: match_barcode_pass' :match / :unknown / :ambiguous
 * (classification.jl:805-824) folded over both passes (:879-897) */
typedef enum bdx_read_status {
    BDX_MATCH = 0,
    BDX_UNKNOWN = 1,   /* file "unknown.fastq[.gz]" */
    BDX_AMBIGUOUS = 2  /* file "ambiguous_classification.fastq[.gz]" */
} bdx_read_status;

/* DynamicRange (classification.jl:9-14), produced by parse_dynamic_range (:83-94) */
typedef struct bdx_range {
    int64_t start_offset;
    int32_t start_from_end;
    int32_t end_from_end;
    int64_t end_offset;
} bdx_range;

/* One barcode set with the per-pass options match_barcode_pass selects
 * (classification.jl:778-792).  Barcodes are the byte strings returned by
 * preprocess_bc_file (fileio.jl:7-72): already B-filtered, upper-cased, U->T,
 * complemented/reversed. */
typedef struct bdx_barcode_set {
    int32_t n_barcodes;
    int32_t trim_side;            /* 0 = nothing, 3, 5  (core.jl:308-313) */
    const uint8_t *bytes;         /* concatenated barcode bytes */
    const int32_t *offsets;       /* n_barcodes + 1 */
    const int32_t *lengths_no_n;  /* bc_lengths_no_N; may be NULL unless has_nindel */
    bdx_range ref_search_range;
    bdx_range barcode_start_range;
    bdx_range barcode_end_range;
} bdx_barcode_set;

/* Hot-path fields of DemuxConfig (classification.jl:16-58). */
typedef struct bdx_params {
    uint32_t struct_size;  /* = sizeof(bdx_params) */
    uint32_t abi_version;  /* = BDX_ABI_VERSION */
    double max_error_rate;
    double min_delta;
    int64_t match, mismatch, indel, nindel;
    int32_t has_nindel;    /* nindel !== nothing */
    int32_t algorithm;     /* bdx_algorithm */
    int32_t is_dual;
    int32_t want_stats;    /* summary=true: alignment positions are tracked for every
                              matched pass (classification.jl:812) and the device keeps
                              the DemuxStats counters */
    bdx_barcode_set set1;
    bdx_barcode_set set2;  /* ignored unless is_dual */
} bdx_params;

/* What worker_task stores per read (core.jl:243-267). */
typedef struct bdx_result {
    int32_t status;     /* bdx_read_status */
    int32_t bc1;        /* 1-based index into set 1; 0 unless status == BDX_MATCH */
    int32_t bc2;        /* 1-based index into set 2 (dual), else 0 */
    int32_t keep_start; /* keep range; -1,-1 when status != BDX_MATCH (=> trim_ranges[i] = */
    int32_t keep_end;   /* nothing, core.jl:250-254); 1,0 = empty keep (classification.jl:932-935) */
} bdx_result;

/* Optional per-pass detail (what match_barcode_pass feeds the stats Dicts,
 * classification.jl:827-865).  score = dist / norm as Float64. */
typedef struct bdx_pass_detail {
    int32_t status; /* bdx_read_status of this pass; -1 = pass not run */
    int32_t bc;
    int32_t dist;   /* integer numerator of the score (weighted distance / mismatches) */
    int32_t norm;   /* normalisation length */
    int32_t start;  /* alignment start / end; -1 when positions were not tracked */
    int32_t end;
} bdx_pass_detail;

typedef struct bdx_config bdx_config;
typedef struct bdx_stream bdx_stream;

const char *bdx_last_error(void);
int bdx_abi_version(void);
/* number of visible CUDA devices (0 if none / driver missing) */
int bdx_device_count(void);

/* Copies everything it needs; the caller keeps ownership of its buffers.
 * Validation mirrors the reference (trim_side in {0,3,5}); additionally rejects
 * what the device encoding cannot express: empty barcodes, zero gap costs
 * (Julia raises DivideError), for :semiglobal and :hamming a max_error_rate
 * whose product with a barcode's length is infinite or outside Int64 (Julia
 * raises InexactError on floor(Int, max_error_rate * length)),
 * |cost| > 2^20, more than 65535 barcodes per set. */
int bdx_config_create(const bdx_params *params, bdx_config **out);
void bdx_config_destroy(bdx_config *cfg);

/* Test / debug hook (not part of the reference boundary): bdx_config_create with single stages of the device
 * pipeline switched off, so that tests can compare the paths against each other.  The results are the same for
 * every flag combination; only the kernels that produce them differ.  The library reads no environment
 * variables. */
enum {
    BDX_DEBUG_NO_FILTER = 1,          /* no bit-parallel kernel: k_literal over every barcode */
    BDX_DEBUG_NO_PREFILTER = 2,       /* no perfect-occurrence / exact-hash tables */
    BDX_DEBUG_NO_SEEDS = 4,           /* no k_seed / k_seed_var levels */
    BDX_DEBUG_NO_SEED_DEEP = 8,       /* no k_seed_deep level */
    BDX_DEBUG_ONE_SEED_LEVEL = 16,    /* only the first seed level */
    BDX_DEBUG_NO_GRAPHS = 32,         /* plain launches instead of CUDA-graph replay of small batches */
    BDX_DEBUG_NO_HAMMING_PACKED = 64, /* :hamming through the edit-distance filter instead of k_hamming_scan */
    BDX_DEBUG_PREFER_SEED_VAR = 128,  /* k_seed_var also for the sets / geometries k_seed's levels take */
    BDX_DEBUG_NO_QGRAM_FILTER = 256   /* k_seed_var verifies every hit (no 3-gram filter in front) */
};
int bdx_config_create_debug(const bdx_params *params, uint32_t debug_flags, bdx_config **out);

/* One per host worker.  Owns three CUDA streams (H2D / kernels / D2H), a ring of
 * BDX_MAX_IN_FLIGHT staging slots (pinned host + device buffers for max_reads reads /
 * max_bytes sequence bytes per batch) and device scratch. */
int bdx_stream_create(const bdx_config *cfg, int device, int32_t max_reads, int64_t max_bytes,
                      bdx_stream **out);
void bdx_stream_destroy(bdx_stream *s);

/* Queue one batch: packed read-1 sequences, raw bytes exactly as read (no case
 * folding; equality is bytewise like codeunits, classification.jl:185).
 * offsets has n_reads + 1 entries, offsets[0] = 0.  Returns after the bytes are in pinned
 * staging, so the caller may reuse its buffers.  At most BDX_MAX_IN_FLIGHT batches may
 * be in flight per stream (BDX_ERR_STATE otherwise). */
int bdx_submit(bdx_stream *s, const uint8_t *seq_bytes, const int32_t *offsets, int32_t n_reads,
               uint64_t tag);
/* Zero-copy variant: borrow the next pinned staging buffers, fill them, commit. */
int bdx_acquire(bdx_stream *s, uint8_t **seq_bytes, int32_t **offsets);
int bdx_commit(bdx_stream *s, int32_t n_reads, uint64_t tag);

/* Like bdx_submit, but the caller guarantees that seq_bytes / offsets are page-locked
 * (bdx_host_alloc or cudaHostRegister) and stay untouched until the batch has been
 * fetched: the H2D copies read them directly, no staging memcpy. */
int bdx_submit_pinned(bdx_stream *s, const uint8_t *seq_bytes, const int32_t *offsets, int32_t n_reads,
                      uint64_t tag);
void *bdx_host_alloc(size_t bytes);
void bdx_host_free(void *p);

/* ---- packed input: half the host->device bytes ---------------------------------------------------------
 * All the path asks of a read byte is whether it equals a barcode byte, so reads may travel as 4-bit codes:
 * 0 = a byte that occurs in no barcode of the config, 1..15 = its distinct barcode bytes (both sets together;
 * bdx_config_code_table).  Layout: byte k of the batch's concatenated reads is nibble k of the packed stream, low
 * nibble first; `offsets` are those of the UNPACKED reads, exactly as for bdx_submit.  The device expands the codes
 * to representative bytes and classifies as usual: the results are identical to bdx_submit on the original bytes.
 * BDX_ERR_INVALID when the config has more than 15 distinct barcode bytes.
 * bdx_pack_reads4 is the host helper a reader calls INSTEAD of copying sequence bytes (AVX2 for letter alphabets;
 * thread-safe, no CUDA): n_bytes input bytes -> (n_bytes + 1) / 2 output bytes. */
int bdx_config_code_table(const bdx_config *cfg, uint8_t table[256]);   /* returns the number of codes incl. 0 */
/* Diagnostics: a text description (one line per table) of what bdx_config_create built for barcode set `pass`
 * (0 or 1) -- which shortcut stages exist and their level parameters (seed lengths, depths, group sizes) -- and a
 * last line `plan: steps=...` naming the kernels the pass launches, in order (k_seed@1 = k_seed's level 1; k_literal
 * @all / @cand / @win / @full / @rest = the reads it scans).  The plan is computed for sm_100's shared-memory limit
 * per block (227 KB), the only device the library runs on.  Writes at most len - 1 bytes and a NUL; returns the
 * full length of the text (0 for an absent second set).  Host data only. */
int bdx_config_describe(const bdx_config *cfg, int pass, char *buf, int len);
int bdx_pack_reads4(const bdx_config *cfg, const uint8_t *seq_bytes, int64_t n_bytes, uint8_t *packed_out);
int bdx_submit_packed4(bdx_stream *s, const uint8_t *packed, const int32_t *offsets, int32_t n_reads, uint64_t tag);
/* like bdx_submit_pinned: packed / offsets are page-locked and stay untouched until the batch has been fetched */
int bdx_submit_packed4_pinned(bdx_stream *s, const uint8_t *packed, const int32_t *offsets, int32_t n_reads,
                              uint64_t tag);

/* ---- search-window input: only the read columns the passes can look at ------------------------------------------
 * A classification depends on a read's length and on its bytes in at most two spans of columns, computed from the
 * length alone: per pass, :semiglobal [start, end] of the resolved search range; :hamming / :exact from its start to
 * min(end, last barcode start) + longest barcode - 1.  A read's "window bytes" are its bytes in those spans, in
 * column order.  Sending them instead of the whole read gives identical results, details and DemuxStats; for long
 * reads with short search ranges it is a small fraction of the bytes.
 * bdx_window_spans: the spans of a read of read_len bases -- lo1, hi1, lo2, hi2 (1-based, inclusive; hi < lo = empty;
 * sorted, merged when they overlap or touch) -- and, as the return value, their total length (< 0: error).
 * bdx_window_reads: the window bytes of a batch (concatenated; win_bytes may be NULL to size the output first) and
 * their offsets win_offsets (n_reads + 1 entries).  offsets are the full reads'.  Both are host-only, thread-safe and
 * need no CUDA device. */
int bdx_window_spans(const bdx_config *cfg, int32_t read_len, int32_t spans[4]);
int bdx_window_reads(const bdx_config *cfg, const uint8_t *seq_bytes, const int32_t *offsets, int32_t n_reads,
                     uint8_t *win_bytes, int32_t *win_offsets);
/* Queue one batch given as window bytes: win / win_offsets as bdx_window_reads makes them, offsets those of the FULL
 * reads exactly as for bdx_submit (max_bytes bounds the full bytes: the device rebuilds them).  packed4 != 0: win is
 * the window stream packed by bdx_pack_reads4 (nibble k = window byte k; win_offsets still count unpacked bytes;
 * BDX_ERR_INVALID when the config has more than 15 distinct barcode bytes).  Before anything is enqueued every
 * read's window length is checked against its length: a mismatch is BDX_ERR_INVALID.  Fetch as usual. */
int bdx_submit_windows(bdx_stream *s, const uint8_t *win, const int32_t *win_offsets, const int32_t *offsets,
                       int32_t n_reads, int packed4, uint64_t tag);
/* like bdx_submit_pinned: win / win_offsets / offsets are page-locked and stay untouched until the batch is fetched */
int bdx_submit_windows_pinned(bdx_stream *s, const uint8_t *win, const int32_t *win_offsets, const int32_t *offsets,
                              int32_t n_reads, int packed4, uint64_t tag);

/* Per-pass details are copied back only when enabled (default: on iff want_stats). */
int bdx_stream_enable_details(bdx_stream *s, int on);

/* Blocks until the oldest in-flight batch is done and copies its results out.
 * details may be NULL; otherwise it receives 2 * n_reads entries laid out
 * [pass][read] (pass 1 block then pass 2 block). */
int bdx_fetch(bdx_stream *s, uint64_t *tag, int32_t *n_reads, bdx_result *results,
              bdx_pass_detail *details);

/* Zero-copy variant of bdx_fetch: pointers into the stream's pinned result staging,
 * valid until BDX_MAX_IN_FLIGHT - 1 further batches have been submitted. */
int bdx_fetch_view(bdx_stream *s, uint64_t *tag, int32_t *n_reads, const bdx_result **results,
                   const bdx_pass_detail **details);

/* submit + fetch of a single batch */
int bdx_classify(bdx_stream *s, const uint8_t *seq_bytes, const int32_t *offsets, int32_t n_reads,
                 bdx_result *results, bdx_pass_detail *details);

/* Device-resident path: inputs and outputs are device pointers on the stream's
 * device; the kernels are enqueued on the stream's compute CUDA stream and the
 * call returns without waiting (bdx_stream_sync waits).  n_reads is not limited
 * by max_reads here, scratch grows on demand.  d_details may be NULL. */
int bdx_classify_device(bdx_stream *s, const uint8_t *d_seq_bytes, const int32_t *d_offsets,
                        int32_t n_reads, bdx_result *d_results, bdx_pass_detail *d_details);
int bdx_stream_sync(bdx_stream *s);
/* cudaStream_t of the compute stream, for callers that record their own events */
void *bdx_stream_cuda_stream(bdx_stream *s);
/* Per-kernel timing of the dominant (bit-parallel semiglobal) kernel: while enabled,
 * every launch of it is bracketed by CUDA events on the compute stream;
 * bdx_stream_profile_read syncs, returns the summed milliseconds and launch count
 * since the last read, and clears the list. */
int bdx_stream_profile(bdx_stream *s, int on);
int bdx_stream_profile_read(bdx_stream *s, double *filter_ms, int32_t *n_launches);
/* The same for every stage: summed milliseconds and launch counts since the last read, indexed
 * [0] k_prefilter [1] k_seed [2] k_seed_deep [3] k_filter [4] k_literal [5] k_hamming_scan / k_seed_hamming
 * [6] k_finalize [7] other.  Clears the list like bdx_stream_profile_read (use one or the other). */
#define BDX_PROFILE_STAGES 8
int bdx_stream_profile_read_stages(bdx_stream *s, double ms[BDX_PROFILE_STAGES], int32_t n_launches[BDX_PROFILE_STAGES]);
/* How many reads (summed over passes) were resolved by the perfect-occurrence prefilter, by the
 * depth-limited seed-and-verify kernel, and how many ran the full-range bit-parallel automaton
 * since the last reset (syncs the stream). */
int bdx_stream_path_counters(bdx_stream *s, int64_t *prefilter_reads, int64_t *seed_reads,
                             int64_t *automaton_reads, int reset);
/* The same three counters plus the work units of the seed kernels (the unit counts of their integer-ALU rooflines,
 * summed over their launches since the last reset):
 *   out[0..2]  prefilter reads, seed reads, automaton reads
 *   out[3]     k_seed_var: window columns it stepped its verified hits over (one bit-parallel column step each)
 *   out[4]     k_seed_var: reads it took in
 *   out[5]     k_seed: q-mers probed (one rolling-hash step and one bitmap test each)
 *   out[6]     k_seed: window columns it verified its hits over
 *   out[7]     k_seed_var: (read, position) pairs scanned (a q-mer code and one or two table look-ups each)
 *   out[8]     k_seed_var: diagonals its 3-gram filter tested
 *   out[9..11] 0 */
int bdx_stream_work_counters(bdx_stream *s, int64_t out[12], int reset);
/* number of kernel launches this stream has issued so far */
int64_t bdx_stream_launch_count(const bdx_stream *s);

/* ---- DemuxStats counters (classification.jl:736-767) ----------------------
 * A flat int64 buffer per stream, accumulated on the device when want_stats:
 *   [0] total  [1] matched  [2] unmatched  [3] ambiguous
 *   sample_counts[(B1+1) * (B2+1)]            index bc1 * (B2+1) + bc2
 *   per pass p in {1,2}:  pos[B_p+1][POS_BINS]  len[B_p+1][LEN_BINS]  dist[B_p+1][DIST_BINS]
 *     row 0 of each is the global histogram, row b the per-barcode one;
 *     pos bin = start + pos_bias (start can be <= 0), len bin = end - start + 1 (up to n + m),
 *     dist bin = integer distance + dist_bias (host converts to round(dist / norm_b, digits=2) keys).
 *     pos/len histograms cover positions up to 1024 bases; a matched pass whose start or length falls
 *     outside goes, exactly, to the stream's overflow list instead (bdx_stats_overflow_fetch) -- long reads
 *     searched near their end.  Its distance is still counted in dist[].
 * bdx_stats_layout describes the offsets; sum the buffers of all streams / GPUs
 * (e.g. one ncclAllReduce(sum, int64)) before converting to DemuxStats. */
typedef struct bdx_stats_layout {
    int64_t total_len;       /* number of int64 entries */
    int64_t sample_off;      /* (B1+1)*(B2+1) entries */
    int32_t b1, b2;          /* set sizes (b2 = 0 when not dual) */
    int32_t pos_bins, len_bins, dist_bins, pos_bias;
    int32_t dist_bias;       /* dist bin = distance + dist_bias (distances are negative when match < 0) */
    int32_t reserved;
    int64_t pos_off[2], len_off[2], dist_off[2];
} bdx_stats_layout;

int bdx_stats_layout_get(const bdx_config *cfg, bdx_stats_layout *out);

/* Report bridge (SURVEY.md section 8f-4): the Dict entries of DemuxStats (classification.jl:736-758) from a
 * counter buffer that has been summed over streams / GPUs.  One entry per non-zero key: pass 1 or 2;
 * kind = position / length / score; bc = 0 for the global Dict (bcN_pos_counts, ...), b >= 1 for
 * bcN_per_bc_*_counts[b]; key for positions and lengths, score = round(dist / norm, digits = 2) for
 * scores (classification.jl:835, :853; equal rounded scores of different distances are merged in the global
 * Dict, exactly as the reference's Dict does).  total / matched / unmatched / ambiguous are counters[0..3],
 * sample_counts is counters[sample_off + bc1 * (b2 + 1) + bc2].  Returns the number of entries (call with
 * out = NULL to size the array), or a negative bdx_status. */
enum { BDX_STATS_POS = 0, BDX_STATS_LEN = 1, BDX_STATS_SCORE = 2 };
typedef struct bdx_stats_entry {
    int32_t pass, kind, bc, reserved;
    int64_t key;
    double score;
    int64_t count;
} bdx_stats_entry;
int64_t bdx_stats_entries(const bdx_config *cfg, const int64_t *counters, bdx_stats_entry *out, int64_t cap);
/* copies the stream's device counters to host (after syncing the stream) */
int bdx_stats_fetch(bdx_stream *s, int64_t *out, int64_t out_len);
/* Matched passes whose start / length did not fit the pos / len histograms: one exact record each.  Returns
 * up to cap records, their total number in *n, and in *lost how many could not be kept (the list holds
 * 2^20 records per stream; lost != 0 means the pos / len Dicts are incomplete).  Concatenate over streams / GPUs. */
typedef struct bdx_stats_overflow {
    int32_t pass;     /* 1 or 2 */
    int32_t bc;       /* 1-based barcode index of that pass */
    int32_t start;    /* alignment start (Dict key of bcN_pos_counts) */
    int32_t length;   /* end - start + 1 (Dict key of bcN_len_counts) */
} bdx_stats_overflow;
int bdx_stats_overflow_fetch(bdx_stream *s, bdx_stats_overflow *out, int64_t cap, int64_t *n, int64_t *lost);
/* device pointer of the counters (for an in-place NCCL all-reduce by the host) */
void *bdx_stats_device_ptr(bdx_stream *s);
int bdx_stats_reset(bdx_stream *s);

/* ---- host-side FASTQ block scanner / packer (SURVEY.md section 8f-1) ---------------------
 * CPU helpers for the data format in front of the hot path; they keep the record semantics
 * of reader_task (core.jl:43-110): a record = four readline()s, each stripping one trailing
 * "\n" or "\r\n"; at end of input missing lines read as "". */
typedef struct bdx_fastq_record {   /* byte ranges inside the scanned buffer, terminators stripped */
    int64_t header_off, seq_off, plus_off, qual_off;
    int32_t header_len, seq_len, plus_len, qual_len;
} bdx_fastq_record;
/* Scans up to max_records records from buf[0, len).  final_block = 0: stop before a record whose
 * four lines are not all terminated inside the buffer (re-present buf + *consumed with the next
 * block); final_block != 0: no data follows, a trailing partial record is completed with empty
 * lines.  Thread-safe; needs no CUDA device. */
int bdx_fastq_scan(const uint8_t *buf, int64_t len, int final_block, int32_t max_records,
                   bdx_fastq_record *recs, int32_t *n_records, int64_t *consumed);
/* Packs the sequence lines of recs[0, n) back to back into seq_out (capacity seq_cap bytes) and
 * writes the n + 1 offsets: exactly the batch layout of bdx_submit / bdx_acquire. */
int bdx_fastq_pack(const uint8_t *buf, const bdx_fastq_record *recs, int32_t n, uint8_t *seq_out,
                   int64_t seq_cap, int32_t *offsets_out);

/* ---- dispatcher over several GPUs (SURVEY.md section 8e) ------------------------------------------
 * Reads are independent, so batches are dealt to streams on the given devices (barcode tables replicated per
 * device, no data-path collective) -- each to the stream with the fewest batches in flight, round-robin among
 * equally loaded ones -- and come back in submission order: what a host that owns the writers needs
 * (core.jl:139-148).  A pool belongs to one thread at a time, like a stream.
 * bdx_pool_submit returns BDX_ERR_STATE when every stream already has BDX_MAX_IN_FLIGHT batches in flight:
 * fetch first.  At most n_devices * streams_per_device * BDX_MAX_IN_FLIGHT batches can
 * be in flight.  bdx_pool_stats_fetch sums the DemuxStats counters of all streams (across processes the
 * host sums the buffers with one all-reduce, see bdx_stats_device_ptr). */
typedef struct bdx_pool bdx_pool;
int bdx_pool_create(const bdx_config *cfg, const int *devices, int n_devices, int streams_per_device,
                    int32_t max_reads, int64_t max_bytes, bdx_pool **out);
void bdx_pool_destroy(bdx_pool *p);
int bdx_pool_submit(bdx_pool *p, const uint8_t *seq_bytes, const int32_t *offsets, int32_t n_reads, uint64_t tag);
int bdx_pool_submit_pinned(bdx_pool *p, const uint8_t *seq_bytes, const int32_t *offsets, int32_t n_reads,
                           uint64_t tag);
int bdx_pool_fetch(bdx_pool *p, uint64_t *tag, int32_t *n_reads, bdx_result *results, bdx_pass_detail *details);
int bdx_pool_fetch_view(bdx_pool *p, uint64_t *tag, int32_t *n_reads, const bdx_result **results,
                        const bdx_pass_detail **details);
int bdx_pool_in_flight(const bdx_pool *p);
int bdx_pool_stats_fetch(bdx_pool *p, int64_t *out, int64_t out_len);

/* ---- host-side barcode-table loader (SURVEY.md section 8f-2) -----------------------------------
 * preprocess_bc_file (fileio.jl:7-72): FASTA when the path ends in .fasta / .fa, otherwise a table
 * (',' for .csv, tab otherwise) with the columns Full_seq, ID, Full_annotation.  Keeps the bases
 * annotated 'B', upper-cases, U -> T, optional complement (ATGCN only) and reversal.  bytes / offsets /
 * lengths_no_n are laid out as bdx_barcode_set wants them and stay valid until the table is destroyed.
 * As in the reference, a FASTA record without sequence lines yields an ID but no sequence, so
 * id_count can exceed count.  Errors (missing file / columns, "Length mismatch between sequence and
 * annotation for ID: ...", fileio.jl:46) return BDX_ERR_INVALID with the text in
 * bdx_barcode_table_error().  Thread-safe; needs no CUDA device. */
typedef struct bdx_barcode_table bdx_barcode_table;
int bdx_barcode_table_load(const char *path, int complement, int rev, bdx_barcode_table **out);
void bdx_barcode_table_destroy(bdx_barcode_table *t);
int32_t bdx_barcode_table_count(const bdx_barcode_table *t);
int32_t bdx_barcode_table_id_count(const bdx_barcode_table *t);
const uint8_t *bdx_barcode_table_bytes(const bdx_barcode_table *t);
const int32_t *bdx_barcode_table_offsets(const bdx_barcode_table *t);       /* count + 1 */
const int32_t *bdx_barcode_table_lengths_no_n(const bdx_barcode_table *t);  /* bc_lengths_no_N */
const char *bdx_barcode_table_id(const bdx_barcode_table *t, int32_t i);
const char *bdx_barcode_table_error(void);

/* ---- device FASTQ block demultiplexer (SURVEY.md section 8f-1 + 8f-3) --------------------------
 * The data formats either side of the hot path, on the device: raw FASTQ text in (the bytes
 * reader_task would split with four readlines per record, core.jl:96-101), and per output file one
 * contiguous run of finished records out -- header, sequence[keep], plus, quality[keep], each
 * followed by "\n" (write_entry, core.jl:135-137; keep range applied as in core.jl:155-173) -- in
 * input order (core.jl:146-148).  The host appends every bucket to its file
 * (prefix "." ids[bc1] ["." ids2[bc2]] ".fastq[.gz]", "unknown...", "ambiguous_classification...",
 * classification.jl:877-900): one write per file and block instead of one per record. */
typedef struct bdx_demux_bucket {
    int32_t status;     /* bdx_read_status: which output file */
    int32_t bc1, bc2;   /* 1-based, 0 = none (as in bdx_result) */
    int32_t n_records;
    int64_t offset1, length1;   /* byte range in out1: the read-1 records (trimmed) */
    int64_t offset2, length2;   /* byte range in out2: the mate records (never trimmed) */
} bdx_demux_bucket;

typedef struct bdx_demux_out {
    int32_t n_records;          /* complete records taken from the block(s) */
    int32_t n_buckets;
    int64_t consumed1, consumed2;   /* bytes of each input covered by those records; re-present the
                                       rest in front of the next block */
    const uint8_t *out1;        /* file-1 records grouped by bucket (NULL in BDX_DEMUX_MATES mode) */
    int64_t out1_len;
    const uint8_t *out2;        /* mate records grouped by bucket (NULL in BDX_DEMUX_SINGLE mode) */
    int64_t out2_len;
    const bdx_demux_bucket *buckets;   /* ascending (status-or-barcode) key order */
    const bdx_result *results;  /* per record, input order */
} bdx_demux_out;

enum {
    BDX_DEMUX_SINGLE = 0,       /* single-end (core.jl:191-196) */
    BDX_DEMUX_MATES = 1,        /* paired, classify_both = false: only file 2 is written, routed by read 1 (:185-190) */
    BDX_DEMUX_BOTH = 2,         /* paired, classify_both = true (:174-184) */
    BDX_DEMUX_DEVICE_IO = 16    /* OR-ed in: fastq1 / fastq2 are device pointers (16-byte aligned) and the
                                   out pointers stay on the device */
};

/* One block of FASTQ text per input file (fastq2 / len2 ignored in BDX_DEMUX_SINGLE mode).  Records
 * are complete when all four lines are terminated inside the block; when the block is the last of
 * its file (single-end: final_block != 0; paired: bit 0 of final_block for file 1, bit 1 for file 2)
 * a truncated last record is completed with empty lines, as `readline` at EOF does.  In the paired
 * modes min(records of file 1, records of file 2) records are taken (`while !eof(io1) && !eof(io2)`,
 * core.jl:48): stop once a final block has been consumed completely.  Blocks must stay below 2^31 bytes.  Synchronous; the pointers in *out
 * belong to the stream and stay valid until its next bdx_demux_block call.  When the config was
 * created with want_stats the DemuxStats counters are updated as by any other classification. */
int bdx_demux_block(bdx_stream *s, const uint8_t *fastq1, int64_t len1, const uint8_t *fastq2, int64_t len2,
                    int final_block, int mode, bdx_demux_out *out);
/* CUDA-event milliseconds of the last bdx_demux_block call: [0] H2D, [1] newline index + records,
 * [2] sequence packing, [3] classification, [4] keys + stable radix sort, [5] offsets + bucket
 * table, [6] record copy, [7] D2H. */
int bdx_demux_stage_ms(const bdx_stream *s, float ms[8]);

/* ---- bench / test utilities (not part of the reference boundary) ----------
 * Synthetic reads of SURVEY.md section 8(d): fixed-length reads over ACGT with a
 * barcode of set 1 (and set 2 when dual) planted after k random edits.  Philox-style
 * counter RNG keyed by (seed, read index): any sub-range can be regenerated
 * independently.  Writes n_reads * read_len bytes and n_reads + 1 offsets. */
typedef struct bdx_synth_spec {
    uint64_t seed;
    int64_t first_read;       /* global index of the first read generated */
    int32_t read_len;
    int32_t plant_permille;   /* probability (per 1000) that set-1 barcode is planted */
    int32_t start_lo, start_hi; /* planted start position range (1-based, inclusive) */
    int32_t n_permille_x10;   /* probability (per 10000) of one base replaced by N */
    int32_t set2_mode;        /* 0 none; 1 set-2 barcode ends end_lo..end_hi bases before the read end;
                                 2 set-2 barcode starts at 1-based position end_lo..end_hi */
    int32_t end_lo, end_hi;
} bdx_synth_spec;
int bdx_synth_reads_device(bdx_stream *s, const bdx_synth_spec *spec, int32_t n_reads,
                           uint8_t *d_seq_bytes, int32_t *d_offsets);

/* Integer-ALU peak microbenchmark (roofline denominator): independent LOP3/IADD3
 * chains at full occupancy on `device`; returns lane-ops per second. */
int bdx_int_alu_peak(int device, double *ops_per_second);

#ifdef __cplusplus
}
#endif
#endif /* BDX_H */
