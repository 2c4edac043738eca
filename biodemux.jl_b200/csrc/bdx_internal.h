// bdx_internal.h -- device-visible parameter blocks shared by the kernels and the
// C-ABI host code of libbdx.  Not installed; include/bdx.h is the public surface.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/bdx.h"

namespace bdx {

constexpr int kMaxBarcodeLen = 256;   // literal kernel DP workspace bound
constexpr int kMaxFilterWords = 2;    // bit-parallel filter: barcodes up to 64 nt
constexpr int kCandMax = 16;          // candidate slots per read and pass
constexpr int kCandOverflow = 255;    // cand_cnt value: scan every barcode
constexpr int kCandWindow = 254;      // cand_cnt value: one candidate, cand[1..2] = read columns that hold all its best alignments
constexpr int kInf = 1 << 29;         // INF_INT stand-in for int32 cells (classification.jl:7)
constexpr int kMaxCost = 1 << 20;

// pass-state codes stored in PassOut.bc when no barcode index applies
constexpr int kBcUnknown = 0;     // :unknown   (classification.jl:806, :821)
constexpr int kBcAmbiguous = -1;  // :ambiguous (classification.jl:823)
constexpr int kBcPending = -2;    // filter kernel left candidates for the literal kernel
constexpr int kBcNotRun = -3;     // pass 2 skipped because pass 1 did not match

// DynamicRange with offsets narrowed to int32 (validated at config creation)
struct DevRange {
    int start_off, start_from_end, end_off, end_from_end;
};

struct SeedLevel {
    int k;                        // edit depth the seeds are complete for (<= allowed)
    int q;                        // seed length (6..12)
    uint32_t pow;                 // kPfBase^(q-1)
    int log2;                     // buckets = 1 << log2
    int bm_log2;                  // first-level bitmap bits = 1 << bm_log2
    int n_entries;
    int max_hits;                 // k_seed: rows of the per-read hit list (reads with more hits go to the next stage)
    const uint32_t *bstart;       // [buckets + 1]
    const uint32_t *entries;      // [n_entries] (barcode index << 8) | seed offset
    const uint32_t *ekeys;        // [n_entries] hash of the entry's q-mer
    const uint32_t *bitmap;
};

// :hamming on 2-bit packed words (hamming.cu): uniform barcode length, <= 4 distinct barcode bytes, no 'N'
struct HammingPacked {
    int enabled;
    int m;                        // the common barcode length (<= 32)
    int allowed;                  // floor(max_error_rate * m)
    int n_seg;                    // allowed + 1 disjoint segments
    int n_bstart;                 // entries of bstart (sum of the segments' buckets + 1 each)
    int seg_off[8], seg_q[8], seg_base[8];   // first base / seed length / first bstart entry of every segment
    const uint16_t *bstart;       // per segment: [4^q + 1] CSR row starts into that segment's entry row
    const uint16_t *entries;      // [n_seg][n_bc] barcode indices grouped by seed code
    const uint2 *bcw;             // [n_bc] the two bit planes of the barcode's 2-bit base codes, base k in bit k
};

// seed-and-verify for variable-length sets / constrained geometries (seed_var.cu): every barcode is cut into
// kdepth[b] + 1 disjoint segments whose first q bases sit in a direct-address table (4^q buckets, 2-bit codes)
struct SeedVar {
    int enabled;
    int q;                        // seed length of table 0
    int q2;                       // seed length of table 1 (0 = one table): segments one base longer use it
    int bstart2;                  // first bstart element of table 1 (= 4^q + 1)
    int n_bstart;                 // elements of bstart: (4^q + 1) [+ (4^q2 + 1)]
    int n_entries;
    int complete;                 // kdepth[b] >= allowed0[b] for every barcode: the candidate sets are supersets
    int group_reads;              // reads a block works on at a time (sized so that their hits fit the block's hit list)
    int hit_rows;                 // hit list capacity in rows of 128 records
    int qgram_filter;             // 3-gram filter in front of the verification: 0 = off, 1 = inside the scan, 2 = over the finished hit list
    double sigma_min;             // min_b (kdepth[b] + 1) / norm[b]: no barcode outside the candidate set scores below
    const uint16_t *bstart;       // [n_bstart] CSR row starts of both tables, absolute indices into entries
    const uint32_t *entries;      // [n_entries] (barcode index << 8) | seed offset
    const uint8_t *kdepth;        // [n_bc] edit depth the barcode's seeds are complete for
};

struct DevSet {
    int n_bc;
    int n_bc_pad;     // n_bc rounded up to a multiple of 32
    int max_m;
    int trim_side;    // 0, 3, 5
    int words;        // 32-bit words per barcode in the filter tables; 0 = no filter for this set
    int n_classes;    // byte classes incl. class 0 = "byte absent from every barcode"
    int use_filter;   // the bit-parallel filter kernel runs for this set (tables exist and the set is not tiny)
    int pad1;
    DevRange rs, bs, be;          // ref_search_range, barcode_start_range, barcode_end_range
    const uint8_t *bc_bytes;      // concatenated barcodes
    const int *bc_off;            // n_bc + 1
    const int *norm;              // normalisation length per barcode (classification.jl:460, :476)
    const uint32_t *peq;          // [words][n_classes][n_bc_pad], barcode rows top-aligned
    const int *filt_allowed;      // [n_bc_pad] unit-cost candidate threshold, -1 = padding
    const int *allowed0;          // [n_bc_pad] floor(max_error_rate * norm) at the initial threshold
    const uint8_t *class_of;      // [256] byte -> class
    // perfect-occurrence prefilter (filter.cu): open-addressing table of barcode q-mer hashes
    int pf_enabled;               // 0 = off (N wildcard rows, barcodes shorter than kPfMinSeed, ...)
    int pf_seed;                  // hashed q-mer length q = min(shortest barcode, kPfMaxSeed)
    uint32_t pf_pow;              // kPfBase^(pf_seed-1)
    int pf_log2;                  // table size = 1 << pf_log2
    int pf_bm_log2;               // bitmap of 1 << pf_bm_log2 bits indexed by the top hash bits
    int pf_stride;                // k_prefilter<0> hashes every pf_stride-th column; the table holds the q-mers at
                                  // offsets 0 .. pf_stride - 1 of every barcode (1: prefixes, every column)
    const uint32_t *pf_bitmap;    // "some barcode q-mer has this hash" (first-level reject)
    const uint32_t *pf_keys;      // [size] hash of the entry's q-mer
    const uint32_t *pf_vals;      // [size] pf_val(barcode, offset, length) (lowest index of identical sequences); kPfEmpty
    const uint8_t *bc_cls;        // barcode bytes mapped through class_of (same offsets as bc_bytes)
    // :semiglobal depth-limited seeds (seed.cu, k_seed): for uniform-length sets, every alignment
    // with <= k edits leaves one of k + 1 disjoint barcode segments intact.  Up to two levels: a
    // shallow one with long, very selective seeds, then the deepest level that is still selective.
    HammingPacked hp;
    int sd_levels;                // 0 = off
    int sd_m;                     // the common barcode length
    SeedLevel sd[2];
    // the deepest level (seed_deep.cu, k_seed_deep): depth sdd_k, segments hashed with their own length --
    // one table per seed length (at most two)
    int sdd_n;                    // 0 = off
    int sdd_k;
    SeedLevel sdd[2];
    int sv_levels;                // 0 = off; level 1 (if any) is the complete one
    int pad3;
    SeedVar sv[2];
};

constexpr int kPfMaxSeed = 12;
constexpr int kPfMinSeed = 6;
constexpr uint32_t kPfBase = 0x9E3779B1u;
constexpr uint32_t kPfMix = 0x85EBCA6Bu;
constexpr uint32_t kPfEmpty = 0xFFFFFFFFu;

__host__ __device__ inline uint32_t pf_slot(uint32_t h, int log2size)
{
    return (h * kPfMix) >> (32 - log2size);
}
// first-level bitmap index.  The polynomial hash keeps its last bytes in the LOW bits, so the top
// bits alone would alias all q-mers that differ only at the end; multiply first.
constexpr uint32_t kPfMix2 = 0xC2B2AE35u;
__host__ __device__ inline uint32_t pf_bit(uint32_t h, int log2bits)
{
    return (h * kPfMix2) >> (32 - log2bits);
}
// hash of a q-mer of a sampled table (pf_stride > 1): its bytes as three little-endian words, the bytes from q on
// zeroed.  k_prefilter<0> reads each sampled q-mer as three words from shared memory; per-column tables keep the
// polynomial hash, which rolls.
__host__ __device__ inline uint32_t pf_words_hash(uint32_t x0, uint32_t x1, uint32_t x2)
{
    return x0 * kPfBase + x1 * kPfMix + x2 * kPfMix2;
}
// pf_vals entry: barcode index (< 65535, so never kPfEmpty), offset of the q-mer in the barcode (< 256) and the
// barcode's length (1 .. 256)
__host__ __device__ inline uint32_t pf_val(int b, int o, int m)
{
    return (uint32_t)b | ((uint32_t)o << 16) | ((uint32_t)(m - 1) << 24);
}
__host__ __device__ inline int pf_val_bc(uint32_t v) { return (int)(v & 0xFFFFu); }
__host__ __device__ inline int pf_val_off(uint32_t v) { return (int)((v >> 16) & 0xFFu); }
__host__ __device__ inline int pf_val_len(uint32_t v) { return (int)(v >> 24) + 1; }

struct DevParams {
    double max_error_rate, min_delta;
    int match, mismatch, indel, nindel, has_n;
    int algo, is_dual, want_stats;
    int unit_costs;   // match 0, mismatch 1, indel 1 (and nindel 1): filter distance is the score
    int two;          // (reserved)
    int debug;        // BDX_DEBUG_* flags of the config (test hooks)
    DevSet set[2];
};

// per read and pass
struct PassOut {
    int bc;     // > 0 matched barcode (1-based) or one of kBc*
    int dist;   // integer score numerator
    int start, end;
};

constexpr int kStatsOvfCap = 1 << 20;   // initial capacity of a stream's overflow list (it is drained / grown, never dropped)
struct StatsDev {
    unsigned long long *buf;  // layout: bdx_stats_layout
    bdx_stats_layout lay;
    bdx_stats_overflow *ovf;  // [ovf_cap] passes whose start / length do not fit the histograms
    unsigned int *n_ovf;      // [2] records appended, records lost (stays 0: the host reserves room per batch)
    unsigned int ovf_cap;
};

struct Scratch {
    PassOut *pass[2];
    uint16_t *cand;       // [n][kCandMax]
    uint8_t *cand_cnt;    // [n]
    int *worklist;        // [n] reads the prefilter left for the next stage
    int *n_work;          // [1]
    int *worklist2;       // [n] reads the seed kernel left for the bit-parallel kernel
    int *n_work2;         // [1]
    int *wl_win;          // [n] seed winners queued for k_literal with a column window
    int *wl_full;         // [n] reads k_filter queued for k_literal with candidate lists
    int *n_lit;           // [2] lengths of wl_win, wl_full
};

// Resident blocks per SM of `kern` with `threads` threads and `smem` bytes of dynamic shared memory on the
// current device; raises the kernel's dynamic shared-memory limit on first use.  Cached per (device, kernel,
// threads, smem): the two runtime queries cost microseconds each, which adds up for 4000-read batches.
cudaError_t blocks_per_sm_cached(const void *kern, int threads, size_t smem, int *per_sm);
// Grid of `kern` for `groups` units of work (blocks' worth of reads): as many blocks as are resident on the device's
// `sm_count` SMs at once, fewer when there is less work, at least one.  Blocks loop over the groups past the grid.
cudaError_t resident_grid(const void *kern, int threads, size_t smem, long long groups, int sm_count, int *blocks);

// dynamic shared memory of each kernel's launch, from its file's layout arithmetic (the pass plan, plan.cu, holds
// them against its budgets)
size_t hamming_scan_smem(const DevSet &S);
size_t prefilter_smem_bytes(const DevSet &S);
int prefilter_blocks_per_sm(size_t smem);   // k_prefilter's resident blocks on sm_100 by shared memory alone
size_t filter_smem_bytes(const DevSet &S);
size_t seed_smem(const DevSet &S, const SeedLevel &L);
size_t deep_smem(const DevSet &S);
size_t seed_var_smem(const DevSet &S, const SeedVar &V);

// ---- launch wrappers (kernels.cu / filter.cu) ----
cudaError_t launch_literal(const DevParams &P, int pass, int from_filter, const uint8_t *seq,
                           const int *off, int n, const Scratch &sc, cudaStream_t st, const int *list = nullptr,
                           const int *n_list = nullptr);   // list: compacted read indices (length on the device)
cudaError_t launch_filter(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                          const Scratch &sc, int sm_count, unsigned long long *counters, const int *wl, const int *n_wl,
                          cudaStream_t st);   // wl: the reads to scan (nullptr: all of them)
// level `level` over the reads of wl_in; the reads it cannot finish are appended to wl_out
cudaError_t launch_seed(const DevParams &P, int pass, int level, const uint8_t *seq, const int *off, int n,
                        const Scratch &sc, const int *wl_in, const int *n_in, int *wl_out, int *n_out, int sm_count,
                        unsigned long long *counters, cudaStream_t st);
// reads of a worklist that no kernel resolved: queue them for k_literal over every barcode
cudaError_t launch_mark_pending(const DevParams &P, int pass, int n, const Scratch &sc, const int *wl, const int *n_wl,
                                cudaStream_t st);
cudaError_t launch_seed_var(const DevParams &P, int pass, int level, const uint8_t *seq, const int *off, int n, const Scratch &sc,
                            const int *wl_in, const int *n_in, int *wl_out, int *n_out, int sm_count,
                            unsigned long long *counters, cudaStream_t st);
cudaError_t launch_seed_deep(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n, const Scratch &sc,
                             const int *wl_in, const int *n_in, int *wl_out, int *n_out, int sm_count,
                             unsigned long long *counters, cudaStream_t st);
cudaError_t launch_prefilter(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                             const Scratch &sc, int sm_count, unsigned long long *counters, cudaStream_t st);
cudaError_t launch_hamming_scan(const DevParams &P, int pass, const uint8_t *seq, const int *off, int n,
                                const Scratch &sc, int sm_count, cudaStream_t st);
cudaError_t launch_finalize(const DevParams &P, const int *off, int n, const Scratch &sc,
                            bdx_result *res, bdx_pass_detail *det, StatsDev stats, cudaStream_t st);
cudaError_t launch_unpack4(const uint8_t *d_packed, uint8_t *d_seq, const int *d_off, int n_reads, long long max_bytes,
                           const uint8_t rep[16], int sm_count, cudaStream_t st);
// search-window input (windows.cu): window bytes (or their 4-bit codes) -> the batch's full-length sequence buffer
cudaError_t launch_expand_windows(const uint8_t *d_win, bool packed, const int *d_win_off, const int *d_off,
                                  uint8_t *d_seq, int n_reads, long long bytes, const DevParams &P, const uint8_t rep[16],
                                  int sm_count, cudaStream_t st);
cudaError_t launch_synth(const DevParams &P, const bdx_synth_spec &spec, int n, uint8_t *seq, int *off,
                         cudaStream_t st);
cudaError_t run_int_alu_peak(int device, double *ops_per_second);

}  // namespace bdx
